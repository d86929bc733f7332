/* jpezy_b200.h -- C ABI of the B200-native baseline-JPEG hot path behind falgon/jpezy's
 * encoder / decoder classes.
 *
 * Every entry point names the reference interface it replaces (paths relative to the reference
 * tree).  Plain pointers and sizes only; no C++/torch types.  Pointers named d_* are device
 * pointers on the context's device, `stream` is a cudaStream_t passed as void* (NULL = the
 * context's own stream).  Host-pointer entry points synchronise before returning; *_dev entry
 * points only enqueue work (results such as byte counts are written to device memory).
 *
 * There is NO CPU fallback: without a usable CUDA device jpezyb200_ctx_create fails with
 * JPEZYB200_ENODEVICE and nothing else can be called.
 */
#ifndef JPEZY_B200_H
#define JPEZY_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define JPEZYB200_API __attribute__((visibility("default")))
#else
#define JPEZYB200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define JPEZYB200_ABI_VERSION 1

/* status codes (reference: C++ exceptions / empty optional, SURVEY.md 8b "Errors") */
enum {
    JPEZYB200_OK = 0,
    JPEZYB200_EINVAL = 1,       /* bad argument (null pointer, zero size, > 65535)                 */
    JPEZYB200_ECAPACITY = 2,    /* output buffer too small (reference: bofstream overflow)         */
    JPEZYB200_ECUDA = 3,        /* CUDA runtime error, see jpezyb200_last_error                   */
    JPEZYB200_ENCCL = 4,        /* multi-GPU exchange impossible (jpezyb200_group_create: no peer access to rank 0) */
    JPEZYB200_ECORRUPT = 5,     /* entropy-coded segment cannot be decoded (reference: decode()
                                   returns an empty optional, src/decoder/jpezy_decoder.hpp:109-114) */
    JPEZYB200_ENODEVICE = 6,    /* no CUDA device: there is no CPU path                            */
    JPEZYB200_ENOMEM = 7,
    JPEZYB200_EUNSUPPORTED = 8, /* frame layout outside what the device decoder handles; from the
                                   decode entry points also per image: a DC coefficient (predictor
                                   plus differences) leaves the int16 range of the coefficient
                                   format.  The reference keeps it in an int and decodes such a
                                   stream; the device reports it instead of a wrapped result.    */
    JPEZYB200_EAGAIN = 9        /* *_dev decode only (reported per image in d_status): the parallel
                                   Huffman decoder did not reach its fixed point within the enqueued
                                   rounds; decode again with JPEZYB200_OPT_SYNC_ROUNDS = 0.  The
                                   host-pointer entry point jpezyb200_decode does that by itself.   */
};

typedef struct jpezyb200_ctx jpezyb200_ctx;

/* One context per device; owns the device scratch (coefficients, bit lengths, scan state, the
 * un-stuffed stream) and one stream.  Used by one host thread at a time. */
JPEZYB200_API int jpezyb200_ctx_create(int device, jpezyb200_ctx** out);
JPEZYB200_API void jpezyb200_ctx_destroy(jpezyb200_ctx* ctx);
JPEZYB200_API const char* jpezyb200_strerror(int code);
JPEZYB200_API const char* jpezyb200_last_error(const jpezyb200_ctx* ctx);
JPEZYB200_API int jpezyb200_abi_version(void);

/* options */
enum {
    JPEZYB200_OPT_PAD_ONES = 1,   /* fill bits of the last scan byte: 1 (default, T.81 F.1.2.3) or 0.
                                     Replaces the padding decision inside srook::io::jpeg::bofstream
                                     (call site src/encoder/jpezy_writer.hpp:101-105). */
    JPEZYB200_OPT_TRANSFORM = 2,  /* forward/inverse transform kernels: 0 = fast path with
                                     guard band + exact recompute (default), 1 = FP64 separable
                                     (validation build); same results.  Other values: EINVAL        */
    JPEZYB200_OPT_BATCH_GROUP_BYTES = 4, /* jpezyb200_encode_batch / decode_batch: host<->device bytes per pipeline stage
                                     (default 96 MiB; images per group = value / (3 * pixels), at least 1)      */
    JPEZYB200_OPT_SHARD_SCRATCH_BYTES = 5, /* jpezyb200_shard_encode_*: bytes of device scratch for this rank's un-stuffed bits;
                                     0 (default) = the reference's own bound, 3 bytes per pixel of the shard.  A shard that does
                                     not fit makes EVERY rank report overflow in phase D (no silently short segment) */
    JPEZYB200_OPT_SYNC_GUESSES = 6, /* decoder, first self-synchronisation launch: 0 (default) = one guessed state per subsequence;
                                     1 = on inputs too small to fill the device (a single frame) one chain per block position of
                                     the MCU, all at once: shortest latency of ONE decode (a 1080p frame: -11 %), six times the
                                     work -- with several decodes in flight on other contexts the default is faster */
    JPEZYB200_OPT_SYNC_ROUNDS = 3, /* self-synchronisation launches enqueued after the first one by the
                                     decoder: n > 0 = exactly n, no host round trip (default 3; the first launch checks
                                     the boundaries of its thread blocks itself, so on ordinary streams none of them has work and
                                     all return at once); 0 = the host polls a device flag after every launch until the fixed
                                     point */
    JPEZYB200_OPT_RESTART_INTERVAL = 7 /* encoders: MCUs per restart interval, 0..65535 (other values: EINVAL); 0 (default) =
                                     no restart markers.  Applies to every single-context encode: jpezyb200_encode,
                                     _encode_batch, _encode_batch_dev, _entropy_encode_dev and the three *_optimized* forms.
                                     The segment then holds the RSTn markers: interval i >= 1 is preceded by FF D((i-1) mod 8),
                                     no marker follows the last one; every interval ends on a byte boundary padded as
                                     JPEZYB200_OPT_PAD_ONES says, and its DC predictors start at 0 (T.81 F.1.2.3, E.1.4).
                                     scan_bytes counts the stuffed bytes, markers included; scan_bits the Huffman-coded bits
                                     only (no padding, no markers).  The file needs a DRI segment (FF DD 00 04 Ri) in front of
                                     SOS (jpezy::jpezy_writer::write_header does that), and jpezyb200_frame.restart_interval to
                                     decode it.  The MCU-row sharded encoders and jpezyb200_group_encode write restart-less
                                     segments only: with a non-zero interval they return JPEZYB200_EUNSUPPORTED. */
};
JPEZYB200_API int jpezyb200_set_option(jpezyb200_ctx* ctx, int option, int64_t value);

/* statistics (monotonic counters since context creation) */
enum {
    JPEZYB200_STAT_KERNEL_LAUNCHES = 1,  /* number of kernels this library launched              */
    JPEZYB200_STAT_GUARD_FWD = 2,        /* DCT coefficients re-computed in exact reference order */
    JPEZYB200_STAT_GUARD_INV = 3,        /* IDCT samples re-computed in exact reference order     */
    JPEZYB200_STAT_SYNC_ROUNDS = 4,      /* self-synchronisation rounds of the last decode        */
    JPEZYB200_STAT_SYNC_ITERS0 = 5,      /* last decode: most shared-memory iterations any CTA needed in launch 0 */
    JPEZYB200_STAT_SYNC_ITERS1 = 6       /* ... and in launch 1 (= synchronisation distance in subsequences)      */
};
JPEZYB200_API int jpezyb200_get_stat(jpezyb200_ctx* ctx, int stat, uint64_t* value);

/* ------------------------------------------------------------------------------------------------
 * Encoder.  Replaces the MCU loop of jpezy::encoder<T>::encode<MODE>()
 * (src/encoder/jpezy_encoder.hpp:55-67: make_YCC :90-144, DCT :146-166, quantization :168-172,
 * encode_huffman :174-225, make_MCU :227-242) together with the bit writer it drives
 * (srook::io::jpeg::bofstream, call sites :189-220).  Produces ONLY the entropy-coded segment
 * (byte-stuffed, last byte padded); the 644-byte header (src/encoder/jpezy_writer.hpp:20-94)
 * and EOI (:101-105) stay with the host writer.
 *
 * r,g,b: planar 8-bit samples, W*H each, row stride W (src/encoder/jpezy_encoder.hpp:105).
 * gray != 0 selects GRAY_MODE (:60-64: Cb/Cr blocks zeroed after colour conversion).
 * ---------------------------------------------------------------------------------------------- */
JPEZYB200_API int jpezyb200_encode(jpezyb200_ctx* ctx, const uint8_t* r, const uint8_t* g, const uint8_t* b, uint32_t W, uint32_t H,
                     int gray, uint8_t* scan_out, size_t scan_cap, size_t* scan_bytes, uint64_t* scan_bits);

/* Batch of nimg images of identical geometry, everything device resident.  Image i reads planes
 * at d_r + i*W*H (etc.) and writes its segment at d_scan + i*slot_bytes; d_scan_bytes[i] /
 * d_scan_bits[i] (device, may be NULL) receive the stuffed byte count / the un-stuffed bit count.
 * A segment that does not fit in slot_bytes sets d_scan_bytes[i] = UINT64_MAX. */
JPEZYB200_API int jpezyb200_encode_batch_dev(jpezyb200_ctx* ctx, const uint8_t* d_r, const uint8_t* d_g, const uint8_t* d_b, uint32_t W,
                               uint32_t H, uint32_t nimg, int gray, uint8_t* d_scan, size_t slot_bytes,
                               uint64_t* d_scan_bytes, uint64_t* d_scan_bits, void* stream);

/* Stuffed byte counts of a device-resident batch on the host: copies n values of d_values (d_scan_bytes or
 * d_scan_bits of jpezyb200_encode_batch_dev / jpezyb200_entropy_encode_dev) into h_out through pinned memory of
 * the context and returns when they have arrived -- i.e. when everything enqueued on `stream` before the call has
 * finished.  This is the one host round trip of a device-resident encode -> decode chain: the decoder entry points
 * take the segment lengths from the host (a JPEG decoder is handed a file of known size,
 * src/decoder/jpezy_decoder.hpp:76-90), the encoder produces them on the device (bofstream's write cursor,
 * src/encoder/jpezy_encoder.hpp:41-45,101-105). */
JPEZYB200_API int jpezyb200_read_sizes(jpezyb200_ctx* ctx, const uint64_t* d_values, uint32_t n, uint64_t* h_out, void* stream);

/* Batch of nimg images in HOST memory (image i: planes at r + i*W*H, segment at scan_out + i*slot_bytes, scan_bytes[i] = its
 * length, UINT64_MAX when it did not fit).  Pipelined over three streams: the host->device copies of one group of images,
 * the kernels of the previous group and the device->host copies of the one before overlap (pin the host buffers for the
 * copies to be asynchronous).  The reference has no batch entry point: this is its encoder::encode() called nimg times
 * (src/encoder/encode_io.hpp:163-165) with the PCIe transfers hidden.  Synchronises before returning. */
JPEZYB200_API int jpezyb200_encode_batch(jpezyb200_ctx* ctx, const uint8_t* r, const uint8_t* g, const uint8_t* b, uint32_t W, uint32_t H,
                           uint32_t nimg, int gray, uint8_t* scan_out, size_t slot_bytes, uint64_t* scan_bytes);

/* One Huffman table as a DHT segment carries it: written by the optimised encoders below, read by the decoders. */
typedef struct jpezyb200_huff {
    uint8_t present;
    uint8_t bits[16];   /* number of codes of length 1..16 (DHT, src/decoder/jpezy_decoder.hpp:208-211) */
    uint8_t vals[256];  /* symbol values in code order (:240)                                         */
} jpezyb200_huff;

/* Optimised Huffman tables (the counterpart of libjpeg's -optimize; the reference has none).  The same encodes as
 * jpezyb200_encode, jpezyb200_encode_batch_dev and jpezyb200_entropy_encode_dev, but every image is coded with Huffman
 * tables fitted to its own symbol counts (T.81 section K.2, code lengths limited to 16, no all-1-bits code word) instead
 * of the Annex K tables K.3-K.6: the same coefficients and decoded pixels in a smaller segment.  The counts and the
 * tables are computed on the device; nothing waits for the host in between.
 *
 * ht / d_ht: [class 0=DC,1=AC][0=luma (Y), 1=chroma (Cb and Cr)] records with present = 1.  They take the place of the
 * DHT contents that the host writer emits from the Annex K tables (write_header, src/encoder/jpezy_writer.hpp:20-94,
 * src/encoder/huffman_table.hpp): copy them into the file's four DHT segments to write it, and into
 * jpezyb200_frame.ht[c][i] (jpezyb200_default_frame's td = {0,1,1}) to decode it.  d_ht is a device array of
 * [nimg][2][2] records.  jpezyb200_encode_optimized reads the sizes and the tables back in one copy; it synchronises
 * as often as jpezyb200_encode.  The MCU-row sharded encoders and jpezyb200_encode_batch have no optimised form.
 * With JPEZYB200_OPT_RESTART_INTERVAL set, the tables are fitted to the symbols of the restart stream (DC differences
 * against predictors that restart at 0 in every interval). */
JPEZYB200_API int jpezyb200_encode_optimized(jpezyb200_ctx* ctx, const uint8_t* r, const uint8_t* g, const uint8_t* b, uint32_t W,
                               uint32_t H, int gray, uint8_t* scan_out, size_t scan_cap, size_t* scan_bytes, uint64_t* scan_bits,
                               jpezyb200_huff ht[2][2]);
JPEZYB200_API int jpezyb200_encode_batch_optimized_dev(jpezyb200_ctx* ctx, const uint8_t* d_r, const uint8_t* d_g, const uint8_t* d_b,
                               uint32_t W, uint32_t H, uint32_t nimg, int gray, uint8_t* d_scan, size_t slot_bytes,
                               uint64_t* d_scan_bytes, uint64_t* d_scan_bits, jpezyb200_huff* d_ht, void* stream);
JPEZYB200_API int jpezyb200_entropy_encode_optimized_dev(jpezyb200_ctx* ctx, const int16_t* d_coefs, uint32_t W, uint32_t H,
                               uint32_t nimg, int gray, uint8_t* d_scan, size_t slot_bytes, uint64_t* d_scan_bytes,
                               uint64_t* d_scan_bits, jpezyb200_huff* d_ht, void* stream);

/* Stage E1+E2 only: planar RGB -> quantised coefficients, int16, zig-zag order
 * (src/jpezy.hpp:36-45), block order Y0 Y1 Y2 Y3 Cb Cr per MCU, MCUs row-major
 * (src/encoder/jpezy_encoder.hpp:227-242).  d_coefs holds nimg * num_mcus * 6 * 64 int16. */
JPEZYB200_API int jpezyb200_transform_fwd_dev(jpezyb200_ctx* ctx, const uint8_t* d_r, const uint8_t* d_g, const uint8_t* d_b,
                                uint32_t W, uint32_t H, uint32_t nimg, int gray, int16_t* d_coefs, void* stream);

/* Stage E3 only: coefficients (layout above) -> stuffed, padded entropy segment(s)
 * (src/encoder/jpezy_encoder.hpp:174-225).  Byte-identical to the reference given identical
 * coefficients (with JPEZYB200_OPT_RESTART_INTERVAL = 0). */
JPEZYB200_API int jpezyb200_entropy_encode_dev(jpezyb200_ctx* ctx, const int16_t* d_coefs, uint32_t W, uint32_t H, uint32_t nimg,
                                 int gray, uint8_t* d_scan, size_t slot_bytes, uint64_t* d_scan_bytes,
                                 uint64_t* d_scan_bits, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Decoder.  Replaces the MCU loop of jpezy::decoder<BuildMode>::decode<MODE>()
 * (src/decoder/jpezy_decoder.hpp:107-130: decode_mcu :504-528, decode_huffman :583-642,
 * inverse_quantization :645-650, inverse_dct :652-670, make_rgb :531-578) and the bit reader
 * (srook::io::jpeg::bifstream, call sites :589,612,634).  Marker parsing (:171-502) stays on the
 * host and hands its result over in jpezyb200_frame.
 * ---------------------------------------------------------------------------------------------- */
typedef struct jpezyb200_frame {
    uint32_t width, height;        /* SOF0 (src/decoder/jpezy_decoder.hpp:286-289)                    */
    uint8_t sample_precision;      /* 8                                                               */
    uint8_t ncomp;                 /* 1 or 3                                                          */
    uint8_t hs[3], vs[3], tq[3];   /* Frame_component H, V, Tq (src/decoder/tables.hpp:18-21); on the
                                      device: luma H, V in {1, 2}, chroma 1x1                         */
    uint8_t td[3], ta[3];          /* Scan_component Td, Ta (:23-26); the reference uses Td for both  */
    uint16_t restart_interval;     /* DRI (src/decoder/jpezy_decoder.hpp:400-404): MCUs per restart
                                      interval, 0 = none                                              */
    uint16_t qt[4][64];            /* natural order, as analyze_dqt stores them (:258-277)            */
    jpezyb200_huff ht[2][4];       /* [class 0=DC,1=AC][id]                                           */
} jpezyb200_frame;

/* Length of each output plane exactly as the reference sizes it
 * (src/decoder/jpezy_decoder.hpp:94-101): (v_unit*vmax*8) * (h_unit*hmax*8). */
JPEZYB200_API size_t jpezyb200_plane_bytes(const jpezyb200_frame* f);
/* Fill a frame descriptor with the layout and Annex K tables jpezy's own encoder writes. */
JPEZYB200_API int jpezyb200_default_frame(uint32_t W, uint32_t H, jpezyb200_frame* f);

/* scan: entropy-coded segment (everything after the SOS header; a trailing EOI marker is allowed).
 * r,g,b: planes of plane_bytes each, row stride = width; rows >= height of the last MCU row land in
 * the tail exactly as in make_rgb (:535-553); bytes never written are zero. */
JPEZYB200_API int jpezyb200_decode(jpezyb200_ctx* ctx, const uint8_t* scan, size_t scan_bytes, const jpezyb200_frame* f, int gray,
                     uint8_t* r, uint8_t* g, uint8_t* b, size_t plane_bytes);

/* Batch, device resident, all images share the frame descriptor.  Image i: segment at
 * d_scan + i*slot_bytes with length h_scan_bytes[i] (HOST array: the file length is host knowledge),
 * planes at d_r + i*plane_bytes.  d_status[i] (device, may be NULL) receives 0, JPEZYB200_ECORRUPT, JPEZYB200_EUNSUPPORTED (a DC
 * coefficient outside the int16 range; that image's planes are not the reference's) or JPEZYB200_EAGAIN (the
 * self-synchronising decoder did not reach its fixed point in the enqueued launches: decode that image again with
 * JPEZYB200_OPT_SYNC_ROUNDS = 0, the host-polled loop). */
JPEZYB200_API int jpezyb200_decode_batch_dev(jpezyb200_ctx* ctx, const uint8_t* d_scan, size_t slot_bytes, const uint64_t* h_scan_bytes,
                               uint32_t nimg, const jpezyb200_frame* f, int gray, uint8_t* d_r, uint8_t* d_g, uint8_t* d_b,
                               size_t plane_bytes, int32_t* d_status, void* stream);

/* The same with the segment lengths in DEVICE memory (d_scan_bytes, e.g. the d_scan_bytes output of jpezyb200_encode_batch_dev):
 * a device-resident transcode needs no host round trip between the encoder and the decoder.  The launch is sized for segments
 * of at most max_scan_bytes (1..slot_bytes); an image whose length turns out larger is not decoded and reports
 * JPEZYB200_ECAPACITY in d_status.  The file-length semantics of the reference (src/decoder/jpezy_decoder.hpp:41-72, the
 * decoder owns a file of known size) stay available through the host-array form above. */
JPEZYB200_API int jpezyb200_decode_batch_dev2(jpezyb200_ctx* ctx, const uint8_t* d_scan, size_t slot_bytes, const uint64_t* d_scan_bytes,
                                uint64_t max_scan_bytes, uint32_t nimg, const jpezyb200_frame* f, int gray, uint8_t* d_r, uint8_t* d_g,
                                uint8_t* d_b, size_t plane_bytes, int32_t* d_status, void* stream);

/* Batch in HOST memory, pipelined like jpezyb200_encode_batch: segment i at scan + i*slot_bytes (scan_bytes[i] bytes), planes of
 * image i at r + i*plane_bytes.  status (host, may be NULL) receives 0 or an error code per image (JPEZYB200_EAGAIN never
 * leaves this call: such an image is decoded again with the host-polled loop).  With status == NULL the call returns the first
 * per-image error instead of JPEZYB200_OK. */
JPEZYB200_API int jpezyb200_decode_batch(jpezyb200_ctx* ctx, const uint8_t* scan, size_t slot_bytes, const uint64_t* scan_bytes, uint32_t nimg,
                           const jpezyb200_frame* f, int gray, uint8_t* r, uint8_t* g, uint8_t* b, size_t plane_bytes, int32_t* status);

/* Stage D1 only: segment(s) -> coefficients (layout of jpezyb200_transform_fwd_dev, DC absolute).  d_status as above: an image
 * whose DC leaves the int16 range reports JPEZYB200_EUNSUPPORTED (its DC coefficients are wrapped). */
JPEZYB200_API int jpezyb200_entropy_decode_dev(jpezyb200_ctx* ctx, const uint8_t* d_scan, size_t slot_bytes,
                                 const uint64_t* h_scan_bytes, uint32_t nimg, const jpezyb200_frame* f, int16_t* d_coefs,
                                 int32_t* d_status, void* stream);

/* Stage D2+D3 only: coefficients -> planar RGB. */
JPEZYB200_API int jpezyb200_transform_inv_dev(jpezyb200_ctx* ctx, const int16_t* d_coefs, const jpezyb200_frame* f, uint32_t nimg,
                                int gray, uint8_t* d_r, uint8_t* d_g, uint8_t* d_b, size_t plane_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * One image, several GPUs: the encoder sharded by MCU rows (BASELINE.json config 5).  No counterpart in the
 * reference (single threaded); the OUTPUT is the reference's: one restart-less segment, byte-identical to
 * jpezyb200_encode on the whole image.  One context (one process) per GPU; the four phases are separated by
 * three tiny all-gathers that the caller performs (NCCL through torch.distributed in jpezy_b200/shard.py):
 *
 *   a: transform the shard's MCU rows                 -> d_last_dc[3]   (quantised DC of Y3, Cb, Cr of the last MCU)
 *      all-gather #1; rank k passes rank k-1's record (rank 0: zeros) as d_dc_init: the running predictors
 *      pre_DC[3] of src/encoder/jpezy_encoder.hpp:180-181 crossing the shard boundary
 *   b: code lengths, local scan, bit scatter          -> d_info[2]      {local bit count, first 8 local bits}
 *      all-gather #2 -> d_all_info[nranks][2]
 *   c: global bit base, ownership of aligned bytes, 0xFF count of the owned bytes (byte stuffing depends on the global
 *      byte alignment)                                -> d_out_bytes[1] owned + stuffed bytes of this rank
 *      all-gather #3 -> d_all_bytes[nranks]
 *   d: stuffed bytes written at this rank's byte base straight into d_dst, the stitched stream, which may live on
 *      another GPU (jpezyb200_ipc_*): the stores go over NVLink, there is no staging copy.
 *
 * Planes passed to phase a hold image rows y_origin.. (row stride W); the shard covers MCU rows
 * [mcu_row0, mcu_row0 + mcu_rows) and needs pixel rows mcu_row0*16 .. min(H, (mcu_row0+mcu_rows)*16) - 1.
 * d_total_bytes (may be NULL) receives the length of the whole stream, d_overflow (may be NULL) 1 when it did
 * not fit dst_cap or a rank's scratch.
 * ---------------------------------------------------------------------------------------------- */
JPEZYB200_API int jpezyb200_shard_encode_a(jpezyb200_ctx* ctx, const uint8_t* d_r, const uint8_t* d_g, const uint8_t* d_b, uint32_t W,
                             uint32_t H, uint32_t mcu_row0, uint32_t mcu_rows, uint32_t y_origin, int gray, int32_t* d_last_dc,
                             void* stream);
JPEZYB200_API int jpezyb200_shard_encode_b(jpezyb200_ctx* ctx, const int32_t* d_dc_init, uint64_t* d_info, void* stream);
JPEZYB200_API int jpezyb200_shard_encode_c(jpezyb200_ctx* ctx, const uint64_t* d_all_info, uint32_t rank, uint32_t nranks,
                             uint64_t* d_out_bytes, void* stream);
JPEZYB200_API int jpezyb200_shard_encode_d(jpezyb200_ctx* ctx, const uint64_t* d_all_bytes, uint8_t* d_dst, size_t dst_cap,
                             uint64_t* d_total_bytes, int32_t* d_overflow, void* stream);

/* The same from ONE host thread (a C or C++ host, as the reference is): a group owns one context per rank -- rank k on CUDA
 * device devices[k]; naming a device more than once emulates several ranks on it -- runs the four phases on the ranks' streams
 * and performs the three exchanges itself (peer copies of 12, 16 and 8 bytes ordered with events; no collective library, no
 * host synchronisation before the end).  d_r[k] / d_g[k] / d_b[k]: device pointers on rank k's device holding the pixel rows
 * of that rank's MCU rows (jpezyb200_group_partition: the same split as jpezy_b200/shard.py), row stride W.  The stitched
 * segment lands in d_dst on rank 0's device; the other devices need peer access to it (JPEZYB200_ENCCL from group_create if
 * the hardware refuses).  Blocking; *scan_bytes receives the segment length. */
typedef struct jpezyb200_group jpezyb200_group;
JPEZYB200_API int jpezyb200_group_create(int nranks, const int* devices, jpezyb200_group** out);
JPEZYB200_API void jpezyb200_group_destroy(jpezyb200_group* g);
JPEZYB200_API int jpezyb200_group_size(const jpezyb200_group* g);
JPEZYB200_API const char* jpezyb200_group_last_error(const jpezyb200_group* g);
JPEZYB200_API jpezyb200_ctx* jpezyb200_group_ctx(jpezyb200_group* g, uint32_t rank);
JPEZYB200_API int jpezyb200_group_partition(const jpezyb200_group* g, uint32_t H, uint32_t rank, uint32_t* mcu_row0, uint32_t* mcu_rows);
JPEZYB200_API int jpezyb200_group_encode(jpezyb200_group* g, const uint8_t* const* d_r, const uint8_t* const* d_g, const uint8_t* const* d_b,
                           uint32_t W, uint32_t H, int gray, uint8_t* d_dst, size_t dst_cap, uint64_t* scan_bytes);

/* One image decoded by several GPUs.  The restart-less entropy-coded segment is decoded whole on every rank (replicas:
 * its self-synchronising decoder is latency bound and a byte-range split would have to redistribute the coefficients by MCU
 * row afterwards, SURVEY.md 8e "fall back to replicas for the entropy stage"); dequantisation, IDCT, upsampling and colour
 * conversion (src/decoder/jpezy_decoder.hpp:645-676, 531-578) are sharded by MCU rows: this rank produces pixel rows of MCU
 * rows [mcu_row0, mcu_row0 + mcu_rows) and stores them straight into the full planes d_r/d_g/d_b, which may be mapped from
 * another GPU (jpezyb200_ipc_*).  The rank that owns the last MCU row also clears the planes' tail. */
JPEZYB200_API int jpezyb200_shard_decode_dev(jpezyb200_ctx* ctx, const uint8_t* d_scan, size_t scan_bytes, const jpezyb200_frame* f,
                               int gray, uint32_t mcu_row0, uint32_t mcu_rows, uint8_t* d_r, uint8_t* d_g, uint8_t* d_b,
                               size_t plane_bytes, int32_t* d_status, void* stream);

/* Peer-visible device buffer for the stitched stream: the owning rank allocates and exports a 64-byte CUDA IPC
 * handle, the other ranks (other processes, other GPUs of the box) map it and pass the mapped pointer as d_dst. */
JPEZYB200_API int jpezyb200_ipc_alloc(jpezyb200_ctx* ctx, size_t bytes, void** d_ptr, uint8_t handle[64]);
JPEZYB200_API int jpezyb200_ipc_open(jpezyb200_ctx* ctx, const uint8_t handle[64], void** d_ptr);
JPEZYB200_API int jpezyb200_ipc_close(jpezyb200_ctx* ctx, void* d_ptr);
JPEZYB200_API int jpezyb200_ipc_free(jpezyb200_ctx* ctx, void* d_ptr);

/* Synthetic planar RGB generator (SURVEY.md 8d), pure integer arithmetic, identical to
 * jpezy_b200.synth on the host.  family: 0 = S-photo, 1 = S-noise, 2 = flat/ramps (adversarial). */
JPEZYB200_API int jpezyb200_synth_dev(jpezyb200_ctx* ctx, uint8_t* d_r, uint8_t* d_g, uint8_t* d_b, uint32_t W, uint32_t H,
                        uint32_t nimg, uint32_t first_frame, int family, void* stream);
/* rows y0 .. y0+nrows-1 of frame `frame` of a W-wide image (the shards of one giant image generate their own rows) */
JPEZYB200_API int jpezyb200_synth_rows_dev(jpezyb200_ctx* ctx, uint8_t* d_r, uint8_t* d_g, uint8_t* d_b, uint32_t W, uint32_t y0,
                             uint32_t nrows, uint32_t frame, int family, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* JPEZY_B200_H */

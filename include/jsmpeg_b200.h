/*
 * jsmpeg_b200.h -- C ABI of libjsmpeg_b200.so: a B200 (sm_100a CUDA) implementation of jsmpeg's
 * MPEG-1 video decode path.  Plain pointers and sizes only.
 *
 * Part 1 is EXACTLY the ABI the reference's own native plugin boundary binds -- the 15 functions
 * its WASM build exports (reference src/wasm/mpeg1.h:10-25, export list build.sh:53-67) and its
 * JS glue calls (src/mpeg1-wasm.js:29, 36, 43, 50, 62-69, 75-88, 103-108).  A reference-side
 * binding that loads this library instead of the WASM module gets the same behaviour:
 * same call protocol, same return values, same bit-index semantics, bit-identical planes.
 *
 * Part 2 is our batch extension (not in the reference): N independent streams on one GPU,
 * device-resident planes, one call decodes the next pictures of every stream.
 */
#ifndef JSMPEG_B200_H
#define JSMPEG_B200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------ */
/* Part 1: the reference ABI (src/wasm/mpeg1.h:10-25)                                          */

typedef struct mpeg1_decoder_t mpeg1_decoder_t;

/* src/wasm/buffer.h:8-11 */
typedef enum {
	BIT_BUFFER_MODE_EVICT = 1,
	BIT_BUFFER_MODE_EXPAND = 2
} bit_buffer_mode_t;

/* mpeg1.h:12 / mpeg1.c:777-782.  Never fails and never takes the process down: without a usable
 * CUDA device (or after any CUDA error later on) the decoder is DEAD -- decode() returns false like
 * "no sequence header yet", writes are swallowed, jsmpeg_b200_decoder_last_error says why (the
 * reason is also printed to stderr once).  Uses the CUDA device set with
 * jsmpeg_b200_set_default_device, else the one named by the environment variable
 * JSMPEG_B200_DEVICE, else device 0. */
mpeg1_decoder_t *mpeg1_decoder_create(unsigned int buffer_size, bit_buffer_mode_t buffer_mode);
/* mpeg1.h:13 / mpeg1.c:784-798 */
void mpeg1_decoder_destroy(mpeg1_decoder_t *self);
/* mpeg1.h:14 / mpeg1.c:800-802, buffer.c:48-65: room for byte_size more bytes (EXPAND: grows;
 * EVICT: discards consumed bytes, buffer.c:167-190); the pointer is HOST memory (pinned) and ALWAYS
 * covers byte_size bytes -- where the reference's own sizing (buffer.c:53-57) would not, the buffer
 * grows to length + byte_size (csrc/bitbuffer.h). */
void *mpeg1_decoder_get_write_ptr(mpeg1_decoder_t *self, unsigned int byte_size);
/* mpeg1.h:15-16 / mpeg1.c:804-810: read position in BITS */
int mpeg1_decoder_get_index(mpeg1_decoder_t *self);
void mpeg1_decoder_set_index(mpeg1_decoder_t *self, unsigned int index);
/* mpeg1.h:17 / mpeg1.c:812-819: commits the bytes; parses the first sequence header */
void mpeg1_decoder_did_write(mpeg1_decoder_t *self, unsigned int byte_size);

/* mpeg1.h:19-23 / mpeg1.c:821-839 */
int mpeg1_decoder_has_sequence_header(mpeg1_decoder_t *self);
float mpeg1_decoder_get_frame_rate(mpeg1_decoder_t *self);
int mpeg1_decoder_get_coded_size(mpeg1_decoder_t *self);
int mpeg1_decoder_get_width(mpeg1_decoder_t *self);
int mpeg1_decoder_get_height(mpeg1_decoder_t *self);
/* mpeg1.h:24-26 / mpeg1.c:841-851: planes of the most recently decoded picture, HOST-visible
 * (pinned), coded size (stride = coded width, coded width / 2); borrowed until the next decode. */
void *mpeg1_decoder_get_y_ptr(mpeg1_decoder_t *self);
void *mpeg1_decoder_get_cr_ptr(mpeg1_decoder_t *self);
void *mpeg1_decoder_get_cb_ptr(mpeg1_decoder_t *self);
/* mpeg1.h:27 / mpeg1.c:853-864: false = no sequence header yet or no picture start code in the
 * buffer; true otherwise (also for skipped B/D pictures).  Synchronous: the planes are complete
 * and host-visible when it returns. */
bool mpeg1_decoder_decode(mpeg1_decoder_t *self);

/* ------------------------------------------------------------------------------------------ */
/* Part 2: batch extension                                                                      */

typedef struct jsmpeg_b200_batch_t jsmpeg_b200_batch_t;

#define JSMPEG_B200_OUT_DEVICE 0 /* planes stay in HBM (jsmpeg_b200_batch_get_planes)           */
#define JSMPEG_B200_OUT_HOST   1 /* every decoded picture is also copied to pinned host memory  */
#define JSMPEG_B200_OUT_RGBA   2 /* run the fused planar->RGBA epilogue (canvas2d.js:53-122)    */

typedef struct jsmpeg_b200_stats_t {
	uint64_t pictures;            /* decode() == true count                                     */
	uint64_t pictures_decoded;    /* I/P pictures reconstructed                                 */
	uint64_t coded_blocks;
	uint64_t macroblocks;         /* macroblocks written by stage 2                             */
	uint64_t algorithmic_bytes;   /* stage-2 bytes: records + planes written + planes referenced */
	uint64_t es_bytes;            /* bitstream bytes consumed by stage 1                        */
	uint64_t h2d_bytes, d2h_bytes;
	uint64_t kernel_launches;     /* scan + parse + reconstruct (+ rgba) launches               */
	uint64_t recon_launches;
	double parse_ms, recon_ms, scan_ms; /* CUDA-event device time on the launching stream       */
	uint64_t parse_errors;        /* pictures whose slice walk hit an invalid code              */
	double walk_ms;               /* part of parse_ms spent in the walk kernel (1a)             */
	uint64_t lane_walk_pictures;  /* pictures walked by the lane-parallel walk (JSMPEG_B200_WALK=lanes), not its serial fall-back */
} jsmpeg_b200_stats_t;

/* n_streams decoders on CUDA device `device`.  max_slots bounds the pictures parsed ahead
 * (records resident in HBM; cut to what the device can hold); 0 = choose from free memory.
 * Never NULL; a batch without a usable device is dead (see jsmpeg_b200_batch_last_error). */
jsmpeg_b200_batch_t *jsmpeg_b200_batch_create(int n_streams, int device, unsigned int max_slots);
void jsmpeg_b200_batch_destroy(jsmpeg_b200_batch_t *b);
/* NULL while the batch works; otherwise the first failure (a CUDA error text).  A dead batch returns
 * 0 / -1 / false from every call and never touches the device again. */
const char *jsmpeg_b200_batch_last_error(jsmpeg_b200_batch_t *b);
/* Tuning knobs, 0 on success.  "chunk_pictures" G: a parse wave is queued in chunks of G pictures per
 * stream and chunk k is reconstructed while chunk k+1 is being parsed (0 = one chunk, no overlap;
 * default from the environment variable JSMPEG_B200_CHUNK, else 0).  "lookahead": pictures parsed
 * ahead per stream beyond the ones a decode call asks for.
 * "slice_walk" (default 0, or JSMPEG_B200_SLICE_WALK): I/P pictures with at least four slices are parsed by a
 * walk kernel that gives every slice a lane of its own instead of cutting one slice's bits into 32 (streams with a
 * slice per macroblock row); the results are the same bit for bit, only the speed differs.
 * "decode_b" (default 0, or the environment variable JSMPEG_B200_DECODE_B; also honoured by decoders made with
 * mpeg1_decoder_create): the B-PICTURE EXTENSION.  The reference skips B pictures (src/mpeg1.js:181-184:
 * decode() returns true, nothing is rendered) and so does this library by default.  With 1, a B picture is
 * decoded after ISO/IEC 11172-2 from the two most recent I/P pictures; decode() still consumes pictures in
 * CODED order, the planes of a B picture are what get_planes / get_host_planes / the reference ABI's
 * get_{y,cr,cb}_ptr return after it, and jsmpeg_b200_batch_last_picture tells type and temporal_reference so
 * that a player can put pictures into display order.  No reference implementation exists for this part. */
int jsmpeg_b200_batch_set_option(jsmpeg_b200_batch_t *b, const char *name, int value);

/* per-stream twins of the reference ABI */
void *jsmpeg_b200_batch_get_write_ptr(jsmpeg_b200_batch_t *b, int stream, unsigned int byte_size);
void jsmpeg_b200_batch_did_write(jsmpeg_b200_batch_t *b, int stream, unsigned int byte_size);
int jsmpeg_b200_batch_get_index(jsmpeg_b200_batch_t *b, int stream);
void jsmpeg_b200_batch_set_index(jsmpeg_b200_batch_t *b, int stream, unsigned int index);
/* returns has_sequence_header */
int jsmpeg_b200_batch_stream_info(jsmpeg_b200_batch_t *b, int stream, int *width, int *height,
                                  int *coded_size, float *frame_rate);

/* MPEG-TS in, demultiplexed on the GPU (mirror of the reference's host demuxer src/ts.js for a
 * buffer of whole 188-byte packets): the payload of every PES packet with stream id `stream_id`
 * (0xE0 = first video stream, ts.js:213-224) is appended to `stream` exactly as if it had been
 * written with get_write_ptr/did_write.  The buffer need not hold whole packets nor begin on a packet
 * boundary: what a call leaves over is kept for the next one (ts.js:25-41) and a lost sync byte is
 * searched for like the reference does (ts.js:155-189); a PID that a later PES header binds to
 * another stream id stops feeding this stream (ts.js:81-83).  Returns the number of
 * elementary-stream bytes appended (-1: the decoder is dead).  pts_out / offset_out (capacity n_max,
 * may be NULL) receive, per
 * PES packet in stream order, its PTS in 90 kHz ticks (0 if absent) and the byte offset of its
 * payload in the stream's buffer -- the table Decoder.Base.write keeps (src/decoder.js:36-47). */
long jsmpeg_b200_batch_write_ts(jsmpeg_b200_batch_t *b, int stream, const uint8_t *ts, size_t n_bytes, int stream_id,
                                uint64_t *pts_out, uint32_t *offset_out, int n_max, int *n_pes);

/* Make everything written so far resident in HBM and indexed (H2D copy of new bytes + start-code
 * scan).  Called implicitly by decode; exposed so that a benchmark can separate it.  Returns the
 * number of picture start codes currently indexed over all streams. */
long jsmpeg_b200_batch_upload(jsmpeg_b200_batch_t *b);
/* Forget the start-code index and all parsed-ahead records, and rewind every stream to bit 0
 * (the elementary streams stay resident in HBM). */
void jsmpeg_b200_batch_rewind(jsmpeg_b200_batch_t *b);

/* Empty every stream's bit buffer (length = index = 0, planes zeroed) but keep its sequence
 * parameters and all allocations: the state of a decoder that has seen the sequence header and
 * nothing else.  The next write + decode pays the full host->device path again. */
void jsmpeg_b200_batch_reset(jsmpeg_b200_batch_t *b);

/* Equivalent to n_pictures consecutive decode() calls on every stream (streams that run out of
 * pictures simply stop).  Returns the number of decode() calls that returned true. */
long jsmpeg_b200_batch_decode(jsmpeg_b200_batch_t *b, int n_pictures, int flags);

/* Device pointers (HBM) of the most recently decoded picture of a stream; 0 on success. */
int jsmpeg_b200_batch_get_planes(jsmpeg_b200_batch_t *b, int stream, void **y, void **cr, void **cb);
/* Host pointers (pinned) of the most recent picture copied out with JSMPEG_B200_OUT_HOST. */
int jsmpeg_b200_batch_get_host_planes(jsmpeg_b200_batch_t *b, int stream, void **y, void **cr, void **cb);
/* RGBA8888 picture (display size, device memory) of the most recent JSMPEG_B200_OUT_RGBA decode */
int jsmpeg_b200_batch_get_rgba(jsmpeg_b200_batch_t *b, int stream, void **rgba);
/* Synchronous copy of that RGBA picture into caller memory (width * height * 4 bytes). */
int jsmpeg_b200_batch_read_rgba(jsmpeg_b200_batch_t *b, int stream, void *rgba);
/* Synchronous copy of the most recent picture's planes into caller memory (coded size). */
int jsmpeg_b200_batch_read_planes(jsmpeg_b200_batch_t *b, int stream, void *y, void *cr, void *cb);

/* picture_coding_type (1 I, 2 P, 3 B, 4 D) and temporal_reference (ISO 11172-2 2.4.2.5) of the picture the
 * stream's last decode() consumed, decoded or skipped; -1 before the first one.  Either pointer may be NULL. */
int jsmpeg_b200_batch_last_picture(jsmpeg_b200_batch_t *b, int stream, int *picture_type, int *temporal_reference);

void jsmpeg_b200_batch_get_stats(jsmpeg_b200_batch_t *b, jsmpeg_b200_stats_t *out);
void jsmpeg_b200_batch_reset_stats(jsmpeg_b200_batch_t *b);

/* ------------------------------------------------------------------------------------------ */
/* Test hooks (used by tests/ only): run a single stage on caller-provided device-agnostic data */

/* Stage 1 alone: parse the picture whose start code ends at start_byte of `es` (host memory) and
 * copy the records back to host arrays sized mb_size * 16 B and mb_size * 768 B. */
int jsmpeg_b200_debug_parse_picture(const uint8_t *es, uint32_t es_len, uint32_t start_byte,
                                    int mb_width, int mb_height, const uint8_t *intra_q,
                                    const uint8_t *non_intra_q, void *info_out, void *hdr_out,
                                    void *coef_out);
/* Stage 2 alone: reconstruct one picture from host record arrays and host forward planes. */
int jsmpeg_b200_debug_reconstruct(int mb_width, int mb_height, const void *hdr, const void *coef,
                                  const uint8_t *fwd_y, const uint8_t *fwd_cr, const uint8_t *fwd_cb,
                                  uint8_t *cur_y, uint8_t *cur_cr, uint8_t *cur_cb);
/* Stage 2 alone over many pictures of any sizes in ONE launcher call, as the engine makes it (the launcher
 * splits the tasks into launches of its per-launch maximum).  kind = which kernel: */
#define JSMPEG_B200_RECON_PLANES 0 /* I/P picture -> planes          */
#define JSMPEG_B200_RECON_RGBA   1 /* I/P picture -> planes + RGBA   */
#define JSMPEG_B200_RECON_B      2 /* B picture -> planes            */
#define JSMPEG_B200_RECON_RGBA_B 3 /* B picture -> planes + RGBA     */
/* geometry[4 i ..] = mb_width, mb_height, display width, height of task i.  Each task brings host buffers of
 * the same sizes for all tasks: hdr[i] cap_mb * 16 B, coef[i] cap_mb * 768 B, fwd[i] / bwd[i] / cur[i] plane
 * sets (Y | Cr | Cb of the task's coded size, contiguous) of cap bytes, at least the plane set + coded width
 * + 64, and rgba[i] of rgba_cap bytes, at least width * height * 4.  bwd is used by the B kinds, rgba by the
 * RGBA kinds (either may be NULL otherwise).  Every buffer is copied to the device whole and back whole, so
 * that whatever a launch wrote anywhere in it comes back.  0 on success, -1 on bad arguments or a CUDA error. */
int jsmpeg_b200_debug_reconstruct_batch(int kind, int n_tasks, const int32_t *geometry, size_t cap_mb, size_t cap,
                                        size_t rgba_cap, void *const *hdr, void *const *coef, void *const *fwd,
                                        void *const *bwd, void *const *cur, void *const *rgba);

/* NULL while the decoder works, else why it is dead (see mpeg1_decoder_create). */
const char *jsmpeg_b200_decoder_last_error(mpeg1_decoder_t *self);

/* jsmpeg_b200_batch_set_option / jsmpeg_b200_batch_last_picture for a decoder of the reference ABI (which has no
 * option call): "decode_b" switches the B-picture extension on, "lookahead" sets the pictures parsed ahead. */
int jsmpeg_b200_decoder_set_option(mpeg1_decoder_t *self, const char *name, int value);
int jsmpeg_b200_decoder_last_picture(mpeg1_decoder_t *self, int *picture_type, int *temporal_reference);

/* CUDA device for decoders created through the reference ABI from now on (the reference ABI has no
 * device argument; the JS/Python class passes its `device` option here). */
void jsmpeg_b200_set_default_device(int device);

/* Bind the calling thread (and the threads it creates, and the pages it first touches, from now on) to
 * the CPUs of the NUMA node CUDA device `device` hangs off, intersected with its current affinity: a
 * decoder's pinned bit buffer and plane ring should live next to its GPU.  Returns the number of CPUs
 * bound to, 0 when the node is unknown (nothing changed), -1 on error; *node_out (may be NULL) = the node. */
int jsmpeg_b200_bind_host_to_device(int device, int *node_out);

const char *jsmpeg_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif

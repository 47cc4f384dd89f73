/*
 * oracle/mpeg1_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * A CPU restatement of the reference's MPEG-1 video decode path (reference src/mpeg1.js ==
 * src/wasm/mpeg1.c, bit reader src/buffer.js == src/wasm/buffer.c), written in the SAME two-stage
 * shape as the CUDA product so that it pins the stage-1 -> stage-2 record format as well:
 *
 *     oracle_parse_picture()   bitstream/VLC walk of one picture  -> mb_record_t[] + int16 coef[]
 *     oracle_reconstruct()     records + forward planes           -> current planes
 *
 * and the reference's 15-function mpeg1_decoder_* ABI (src/wasm/mpeg1.h:10-25) on top of the two.
 *
 * Pinning: the reference has no tests or golden vectors (SURVEY.md section 4), so this file is
 * pinned by running the reference itself: tests/test_oracle_vs_reference.py compares every plane
 * byte and every bit index against oracle/_ref/libjsmpeg_ref.so (the unmodified reference C,
 * compiled in place) on FFmpeg-encoded clips and on the synthetic syntax-corner streams, and
 * tests/golden/ holds plane checksums produced by that reference build.
 *
 * B pictures.  The reference skips them (mpeg1.js:181-184) and so does this file by default.  With
 * oracle_set_decode_b(1) -- the opt-in extension of the product, SURVEY 8(f) rank 4 -- a B picture is decoded
 * after ISO/IEC 11172-2 (2.4.3.6 macroblock layer, 2.4.4.2/2.4.4.3 skipped macroblocks and bidirectional
 * prediction, table B.2d = the reference's unused MACROBLOCK_TYPE_B, mpeg1.js:1152-1175) with the reference's own
 * building blocks (same bit reader, vector arithmetic, dequantisation, IDCT, flat-index prediction).  PARITY OF
 * THAT PART IS UNPINNED BY THE REFERENCE (there is nothing to run); it is checked against FFmpeg's mpeg1video
 * decoder by PSNR (tests/test_b_pictures.py), which proves the prediction structure, not bit-exactness.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load this library.
 * It deliberately decodes VLCs a different way (bit-by-bit trie built from the ISO-form code
 * lists) than the product (clz-indexed LUTs).
 */
#include <stdbool.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../jsmpeg_b200/csrc/records.h"
#include "vlc_tables_oracle.h"

/* ------------------------------------------------------------------------------------------ */
/* VLC tries                                                                                   */

typedef struct { int16_t child[2]; int value; bool leaf; } trie_node_t;
typedef struct { trie_node_t *nodes; int count; } trie_t;

enum { T_MBA, T_TYPE_I, T_TYPE_P, T_TYPE_B, T_CBP, T_MOTION, T_DC_LUMA, T_DC_CHROMA, T_DCT, T_COUNT };
static trie_t g_trie[T_COUNT];
static bool g_tries_ready = false;
#define VLC_INVALID (-999999)

static void trie_build(trie_t *t, const vlc_code_t *codes) {
	int n = 0, total = 1;
	for (const vlc_code_t *c = codes; c->code; c++) { n++; total += (int)strlen(c->code); }
	t->nodes = (trie_node_t *)calloc(total, sizeof(trie_node_t));
	t->count = 1;
	for (const vlc_code_t *c = codes; c->code; c++) {
		int at = 0;
		for (const char *p = c->code; *p; p++) {
			int b = *p - '0';
			if (!t->nodes[at].child[b]) t->nodes[at].child[b] = (int16_t)t->count++;
			at = t->nodes[at].child[b];
		}
		t->nodes[at].leaf = true;
		t->nodes[at].value = c->value;
	}
}

static void tries_init(void) {
	if (g_tries_ready) return;
	trie_build(&g_trie[T_MBA], ORACLE_MACROBLOCK_ADDRESS_INCREMENT);
	trie_build(&g_trie[T_TYPE_I], ORACLE_MACROBLOCK_TYPE_INTRA);
	trie_build(&g_trie[T_TYPE_P], ORACLE_MACROBLOCK_TYPE_PREDICTIVE);
	trie_build(&g_trie[T_TYPE_B], ORACLE_MACROBLOCK_TYPE_B);
	trie_build(&g_trie[T_CBP], ORACLE_CODE_BLOCK_PATTERN);
	trie_build(&g_trie[T_MOTION], ORACLE_MOTION);
	trie_build(&g_trie[T_DC_LUMA], ORACLE_DCT_DC_SIZE_LUMINANCE);
	trie_build(&g_trie[T_DC_CHROMA], ORACLE_DCT_DC_SIZE_CHROMINANCE);
	trie_build(&g_trie[T_DCT], ORACLE_DCT_COEFF);
	g_tries_ready = true;
}

/* ------------------------------------------------------------------------------------------ */
/* Bit reader over a byte span (MSB first; buffer.js:152-187).  Bytes past the end read as 0,   */
/* which is what a JS typed-array read past byteLength yields after `& mask`.                    */

typedef struct { const uint8_t *bytes; uint32_t length; uint32_t index; /* in bits */ } bits_t;

static inline int bit_at(const bits_t *b, uint32_t i) {
	uint32_t byte = i >> 3;
	return byte < b->length ? (b->bytes[byte] >> (7 - (i & 7))) & 1 : 0;
}
static int bits_read(bits_t *b, int count) {
	int v = 0;
	for (int k = 0; k < count; k++) v = (v << 1) | bit_at(b, b->index + k);
	b->index += count;
	return v;
}
static inline void bits_skip(bits_t *b, int count) { b->index += count; }

/* buffer.js:115-128.  A start code needs its 4 bytes inside the buffer. */
static int bits_find_next_start_code(bits_t *b) {
	for (uint32_t i = (b->index + 7) >> 3; i + 3 < b->length; i++) {
		if (b->bytes[i] == 0 && b->bytes[i + 1] == 0 && b->bytes[i + 2] == 1) {
			b->index = (i + 4) << 3;
			return b->bytes[i + 3];
		}
	}
	b->index = b->length << 3;
	return -1;
}
/* buffer.js:130-139 */
static int bits_find_start_code(bits_t *b, int code) {
	for (;;) {
		int c = bits_find_next_start_code(b);
		if (c == code || c == -1) return c;
	}
}
/* buffer.js:141-150 */
static bool bits_next_bytes_are_start_code(const bits_t *b) {
	uint32_t i = (b->index + 7) >> 3;
	if (i >= b->length) return true;
	return i + 2 < b->length && b->bytes[i] == 0 && b->bytes[i + 1] == 0 && b->bytes[i + 2] == 1;
}

/* mpeg1.js:66-72 readHuffman, as a trie walk.  The reference has no defined result for an
 * invalid code; we return VLC_INVALID and the caller abandons the slice, with the bit index still at the
 * start of that code -- where the search for the next start code then begins (the CUDA walk does the same, so
 * the two agree record for record on damaged streams too; only the reference's own behaviour is undefined there). */
static int read_vlc(bits_t *b, int which) {
	const trie_t *t = &g_trie[which];
	const uint32_t start = b->index;
	int at = 0;
	for (;;) {
		at = t->nodes[at].child[bits_read(b, 1)];
		if (!at) { b->index = start; return VLC_INVALID; } /* (nothing of an invalid code is consumed: the product's rule) */
		if (t->nodes[at].leaf) return t->nodes[at].value;
	}
}

/* ------------------------------------------------------------------------------------------ */
/* Stage 1: picture parse -> records                                                            */

typedef struct {
	int mb_width, mb_size;
	uint8_t intra_q[64], non_intra_q[64]; /* de-zigzagged, mpeg1.js:100-116 */
} seq_params_t;

typedef struct {
	bits_t bits;
	const seq_params_t *seq;
	picture_info_t *info;
	mb_record_t *hdr;
	int16_t *coef;
	int picture_type, full_pel, r_size, f;
	int qscale, mb_addr;
	bool slice_begin;
	int mv_h, mv_v, mv_h_prev, mv_v_prev;
	int dc_pred[3]; /* Y, then the predictor used by block 4, then the one used by block 5 */
	/* B pictures: the backward vector with its own f_code, and how the last macroblock was predicted */
	int full_pel_b, r_size_b, f_b;
	int mvb_h, mvb_v, mvb_h_prev, mvb_v_prev;
	uint8_t last_motion; /* MBF_MOTION_FWD | MBF_MOTION_BWD of the previous macroblock (a skipped one repeats it) */
} parse_t;

static int g_decode_b = 0;
/* the B-picture extension: 0 (default) = B pictures are skipped like the reference does */
void oracle_set_decode_b(int on) { g_decode_b = on; }

static void reset_dc(parse_t *p) { p->dc_pred[0] = p->dc_pred[1] = p->dc_pred[2] = 128; }
static void reset_mv(parse_t *p) {
	p->mv_h = p->mv_v = p->mv_h_prev = p->mv_v_prev = 0;
	p->mvb_h = p->mvb_v = p->mvb_h_prev = p->mvb_v_prev = 0; /* (unused outside B pictures) */
}

static int16_t sat16(int v) { return (int16_t)(v > 32767 ? 32767 : (v < -32768 ? -32768 : v)); }

/* mpeg1.js:698-811 decodeBlock, bitstream part only.  Returns false on an invalid code. */
static bool parse_block(parse_t *p, int mb, int block, bool intra, uint8_t *dc_only_mask) {
	int16_t *out = p->coef + ((size_t)mb * 6 + block) * 64;
	memset(out, 0, 64 * sizeof(int16_t));
	int n = 0;
	const uint8_t *q;
	if (intra) {
		/* mpeg1.js:705-751: DC size VLC, differential, predictor update.  Block 4 uses the
		 * predictor the reference calls "Cr", block 5 the one it calls "Cb" (mpeg1.js:717,739-744). */
		int *pred = &p->dc_pred[block < 4 ? 0 : block - 3];
		int size = read_vlc(&p->bits, block < 4 ? T_DC_LUMA : T_DC_CHROMA);
		if (size == VLC_INVALID) return false;
		int dc = *pred;
		if (size > 0) {
			int diff = bits_read(&p->bits, size);
			if (diff & (1 << (size - 1))) dc += diff;
			else dc += (int)((~0u << size) | (uint32_t)(diff + 1));
		}
		*pred = dc;
		out[0] = sat16(dc * 8); /* x PREMULTIPLIER[0]=32 in stage 2 gives dc<<8, mpeg1.js:747 */
		q = p->seq->intra_q;
		n = 1;
	} else {
		q = p->seq->non_intra_q;
	}

	for (;;) { /* mpeg1.js:757-811 */
		int run, level;
		int coeff = read_vlc(&p->bits, T_DCT);
		if (coeff == VLC_INVALID) return false;
		if (coeff == 0x0001 && n > 0 && bits_read(&p->bits, 1) == 0) break; /* EOB, mpeg1.js:763 */
		if (coeff == 0xffff) { /* escape, mpeg1.js:767-780 */
			run = bits_read(&p->bits, 6);
			level = bits_read(&p->bits, 8);
			if (level == 0) level = bits_read(&p->bits, 8);
			else if (level == 128) level = bits_read(&p->bits, 8) - 256;
			else if (level > 128) level -= 256;
		} else {
			run = coeff >> 8;
			level = coeff & 0xff;
			if (bits_read(&p->bits, 1)) level = -level;
		}
		n += run;
		if (n > 63) { /* JS: ZIG_ZAG[n] is undefined, the store is a no-op (mpeg1.js:790-810) */
			p->info->error = PARSE_ERR_COEF_INDEX;
			n++;
			continue;
		}
		int idx = ORACLE_ZIG_ZAG[n];
		n++;
		/* dequantise, oddify toward zero, clip (mpeg1.js:794-807) */
		level *= 2;
		if (!intra) level += level < 0 ? -1 : 1;
		level = (level * p->qscale * q[idx]) >> 4; /* arithmetic shift: floors negatives */
		if ((level & 1) == 0) level -= level > 0 ? 1 : -1;
		if (level > 2047) level = 2047;
		else if (level < -2048) level = -2048;
		out[idx] = (int16_t)level;
	}
	if (n == 1) *dc_only_mask |= (uint8_t)(0x20 >> block); /* mpeg1.js:838,850 */
	p->info->n_coded_blocks++;
	return true;
}

/* mpeg1.js:395-457, one component */
static bool parse_motion_component_f(parse_t *p, int r_size, int f, int full_pel, int *prev, int *mv) {
	int code = read_vlc(&p->bits, T_MOTION);
	if (code == VLC_INVALID) return false;
	int d = code;
	if (code != 0 && f != 1) {
		int r = bits_read(&p->bits, r_size);
		d = ((abs(code) - 1) << r_size) + r + 1;
		if (code < 0) d = -d;
	}
	*prev += d;
	if (*prev > (f << 4) - 1) *prev -= f << 5;
	else if (*prev < -(f << 4)) *prev += f << 5;
	*mv = full_pel ? *prev * 2 : *prev;
	return true;
}
static bool parse_motion_component(parse_t *p, int *prev, int *mv) {
	return parse_motion_component_f(p, p->r_size, p->f, p->full_pel, prev, mv);
}

static void emit_predicted(parse_t *p, int addr, uint8_t extra_flags) {
	mb_record_t *r = &p->hdr[addr];
	memset(r, 0, sizeof(*r));
	r->mv_h = (int16_t)p->mv_h;
	r->mv_v = (int16_t)p->mv_v;
	r->flags = MBF_PRESENT | extra_flags;
	r->qscale = (uint8_t)p->qscale;
	r->bit_pos = p->bits.index;
	if (p->picture_type == 3) { /* ISO 11172-2 2.4.4.2: same prediction and vectors as the macroblock before */
		r->flags |= p->last_motion;
		if (!(p->last_motion & MBF_MOTION_FWD)) r->mv_h = r->mv_v = 0;
		if (p->last_motion & MBF_MOTION_BWD) r->mv_bwd = ((uint32_t)p->mvb_h & 0xffffu) | ((uint32_t)p->mvb_v << 16);
	}
	p->info->n_present++;
}

/* mpeg1.js:294-392 decodeMacroblock.  Returns false when the slice walk must stop. */
static bool parse_macroblock(parse_t *p) {
	int increment = 0;
	int t = read_vlc(&p->bits, T_MBA);
	while (t == 34) t = read_vlc(&p->bits, T_MBA);                 /* stuffing */
	while (t == 35) { increment += 33; t = read_vlc(&p->bits, T_MBA); } /* escape   */
	if (t == VLC_INVALID) return false;
	increment += t;

	if (p->slice_begin) { /* mpeg1.js:312-317: first increment only positions the address */
		p->slice_begin = false;
		p->mb_addr += increment;
	} else {
		if (p->mb_addr + increment >= p->seq->mb_size) return true; /* mpeg1.js:319-322 (loop goes on) */
		if (increment > 1) { /* mpeg1.js:323-334 */
			reset_dc(p);
			if (p->picture_type == 2) reset_mv(p); /* (B pictures keep their vectors: ISO 11172-2 2.4.4.2) */
		}
		while (increment > 1) { /* skipped macroblocks: predicted copy, mpeg1.js:336-346 */
			p->mb_addr++;
			emit_predicted(p, p->mb_addr, MBF_SKIPPED);
			increment--;
		}
		p->mb_addr++;
	}
	int mb = p->mb_addr;
	if (mb < 0 || mb >= p->seq->mb_size) return false; /* out of the picture: memory safety */

	int type = read_vlc(&p->bits, p->picture_type == 1 ? T_TYPE_I : (p->picture_type == 2 ? T_TYPE_P : T_TYPE_B));
	if (type == VLC_INVALID) return false;
	bool intra = type & 0x01;
	if (type & 0x10) p->qscale = bits_read(&p->bits, 5);

	uint32_t mb_bit_pos = p->bits.index;
	if (intra) {
		reset_mv(p); /* mpeg1.js:363-367 (B: both predictors, ISO 11172-2 2.4.4.3) */
		/* (a skipped macroblock must not follow an intra one in a B picture; if a stream does it anyway it is
		 * predicted forward with the reset, i.e. zero, vector) */
		p->last_motion = MBF_MOTION_FWD;
	} else {
		reset_dc(p); /* mpeg1.js:370-372 */
		if (type & 0x08) {
			if (!parse_motion_component(p, &p->mv_h_prev, &p->mv_h)) return false;
			if (!parse_motion_component(p, &p->mv_v_prev, &p->mv_v)) return false;
		} else if (p->picture_type == 2) {
			reset_mv(p); /* mpeg1.js:452-456 */
		}
		if (p->picture_type == 3) { /* a direction that is not used keeps its predictor */
			if (type & 0x04) {
				if (!parse_motion_component_f(p, p->r_size_b, p->f_b, p->full_pel_b, &p->mvb_h_prev, &p->mvb_h)) return false;
				if (!parse_motion_component_f(p, p->r_size_b, p->f_b, p->full_pel_b, &p->mvb_v_prev, &p->mvb_v)) return false;
			}
			p->last_motion = (uint8_t)(((type & 0x08) ? MBF_MOTION_FWD : 0) | ((type & 0x04) ? MBF_MOTION_BWD : 0));
		}
	}

	int cbp = (type & 0x02) ? read_vlc(&p->bits, T_CBP) : (intra ? 0x3f : 0);
	if (cbp == VLC_INVALID) return false;

	mb_record_t *r = &p->hdr[mb];
	if (!(r->flags & MBF_PRESENT)) p->info->n_present++;
	memset(r, 0, sizeof(*r));
	r->mv_h = (int16_t)p->mv_h;
	r->mv_v = (int16_t)p->mv_v;
	r->flags = MBF_PRESENT | (intra ? MBF_INTRA : 0);
	r->qscale = (uint8_t)p->qscale;
	r->bit_pos = mb_bit_pos;
	if (p->picture_type == 3 && !intra) {
		r->flags |= p->last_motion;
		/* a vector that is not used is stored as zero (the record then does not depend on stale predictors) */
		if (!(p->last_motion & MBF_MOTION_FWD)) r->mv_h = r->mv_v = 0;
		if (p->last_motion & MBF_MOTION_BWD) r->mv_bwd = ((uint32_t)p->mvb_h & 0xffffu) | ((uint32_t)p->mvb_v << 16);
	}
	uint8_t dc_only = 0;
	bool ok = true;
	for (int block = 0; block < 6 && ok; block++) {
		if (cbp & (0x20 >> block)) {
			ok = parse_block(p, mb, block, intra, &dc_only);
			if (ok) r->cbp |= (uint8_t)(0x20 >> block);
		}
	}
	r->dc_only = dc_only;
	return ok;
}

/* mpeg1.js:255-276 decodeSlice */
static void parse_slice(parse_t *p, int slice) {
	p->slice_begin = true;
	p->mb_addr = (slice - 1) * p->seq->mb_width - 1;
	reset_mv(p);
	reset_dc(p);
	p->last_motion = MBF_MOTION_FWD;
	p->qscale = bits_read(&p->bits, 5);
	while (bits_read(&p->bits, 1)) bits_skip(&p->bits, 8);
	do {
		if (!parse_macroblock(p)) {
			if (!p->info->error) p->info->error = PARSE_ERR_INVALID_VLC;
			break;
		}
	} while (!bits_next_bytes_are_start_code(&p->bits));
}

/* mpeg1.js:174-247 decodePicture, bitstream part.  `index` enters just after the picture start
 * code.  hdr[] must be zeroed by the caller (no MBF_PRESENT).  Exported for the tests. */
void oracle_parse_picture(const uint8_t *es, uint32_t es_len, uint32_t start_bit,
                          const seq_params_t *seq, picture_info_t *info,
                          mb_record_t *hdr, int16_t *coef) {
	tries_init();
	parse_t p;
	memset(&p, 0, sizeof(p));
	memset(info, 0, sizeof(*info));
	p.bits.bytes = es; p.bits.length = es_len; p.bits.index = start_bit;
	p.seq = seq; p.info = info; p.hdr = hdr; p.coef = coef;
	info->start_byte = start_bit >> 3;

	bits_skip(&p.bits, 10);
	p.picture_type = bits_read(&p.bits, 3);
	bits_skip(&p.bits, 16);
	info->picture_type = p.picture_type;
	info->status = PIC_IGNORED;
	if (p.picture_type <= 0 || p.picture_type > 3 || (p.picture_type == 3 && !g_decode_b)) { info->end_bit = p.bits.index; return; }
	if (p.picture_type >= 2) {
		p.full_pel = bits_read(&p.bits, 1);
		int f_code = bits_read(&p.bits, 3);
		info->full_pel = p.full_pel; info->f_code = f_code;
		if (f_code == 0) { info->end_bit = p.bits.index; return; }
		p.r_size = f_code - 1;
		p.f = 1 << p.r_size;
	}
	if (p.picture_type == 3) { /* ISO 11172-2 2.4.2.5: full_pel_backward_vector, backward_f_code */
		p.full_pel_b = bits_read(&p.bits, 1);
		int f_code_b = bits_read(&p.bits, 3);
		info->reserved[1] = p.full_pel_b << 4 | f_code_b;
		if (f_code_b == 0) { info->end_bit = p.bits.index; return; }
		p.r_size_b = f_code_b - 1;
		p.f_b = 1 << p.r_size_b;
	}
	info->status = PIC_DECODED;

	int code;
	do { code = bits_find_next_start_code(&p.bits); } while (code == 0xB5 || code == 0xB2);
	while (code >= 0x01 && code <= 0xAF) {
		parse_slice(&p, code);
		code = bits_find_next_start_code(&p.bits);
	}
	if (code != -1) p.bits.index -= 32; /* mpeg1.js:209-213 */
	info->end_bit = p.bits.index;
}

/* ------------------------------------------------------------------------------------------ */
/* Stage 2: records -> planes                                                                   */

/* One 8-point pass of the reference's integer IDCT (mpeg1.js:925-947 / :952-981).  `s` is the
 * element stride; shift = false for the column pass, true for the row pass ((v+128)>>8). */
static void idct_pass(int *v, int s, bool shift) {
	int b1 = v[4 * s];
	int b3 = v[2 * s] + v[6 * s];
	int b4 = v[5 * s] - v[3 * s];
	int t1 = v[1 * s] + v[7 * s];
	int t2 = v[3 * s] + v[5 * s];
	int b6 = v[1 * s] - v[7 * s];
	int b7 = t1 + t2;
	int m0 = v[0];
	int x4 = ((b6 * 473 - b4 * 196 + 128) >> 8) - b7;
	int x0 = x4 - (((t1 - t2) * 362 + 128) >> 8);
	int x1 = m0 - b1;
	int x2 = (((v[2 * s] - v[6 * s]) * 362 + 128) >> 8) - b3;
	int x3 = m0 + b1;
	int y3 = x1 + x2, y4 = x3 + b3, y5 = x1 - x2, y6 = x3 - b3;
	int y7 = -x0 - ((b4 * 473 + b6 * 196 + 128) >> 8);
	int o[8] = { b7 + y4, x4 + y3, y5 - x0, y6 - y7, y6 + y7, x0 + y5, y3 - x4, y4 - b7 };
	for (int k = 0; k < 8; k++) v[k * s] = shift ? (o[k] + 128) >> 8 : o[k];
}

static inline uint8_t clamp255(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

/* mpeg1.js:459-687 copyMacroblock for one plane: `size` x `size` block at (col,row) block units,
 * vector (mh, mv) in half-pel units of that plane.  The source index is FLAT (a vector leaving
 * the row wraps into the neighbouring row, mpeg1.js:479,567).  A tap outside the plane reads
 * `undefined` in JS, the sum becomes NaN and `NaN >> k` is 0, so any out-of-plane tap zeroes the
 * whole output pixel (SURVEY Q11). */
static void predict_plane(uint8_t *dst, const uint8_t *src, int stride, int plane_size,
                          int row, int col, int size, int mh, int mv) {
	int H = mh >> 1, V = mv >> 1, oh = mh & 1, ov = mv & 1;
	int base = (row * size + V) * stride + col * size + H;
	for (int y = 0; y < size; y++) {
		for (int x = 0; x < size; x++) {
			int i = base + y * stride + x;
			int taps[4] = { i, i + 1, i + stride, i + stride + 1 };
			int use[4] = { 1, oh, ov, oh && ov };
			int sum = 0, n = 0; bool inside = true;
			for (int k = 0; k < 4; k++) {
				if (!use[k]) continue;
				if (taps[k] < 0 || taps[k] >= plane_size) { inside = false; break; }
				sum += src[taps[k]]; n++;
			}
			int v = !inside ? 0 : (n == 4 ? (sum + 2) >> 2 : (n == 2 ? (sum + 1) >> 1 : sum));
			dst[(row * size + y) * stride + col * size + x] = (uint8_t)v;
		}
	}
}

typedef struct { uint8_t *y, *cr, *cb; } planes_t;
static void free_planes(planes_t *p) { free(p->y); free(p->cr); free(p->cb); }

/* One macroblock's prediction from one reference into `cur` (the three planes). */
static void predict_macroblock(const seq_params_t *seq, int cw, int ysize, int mb, int mh, int mv,
                               const planes_t *ref, planes_t *cur) {
	int hw = cw >> 1, csize = ysize >> 2;
	int row = mb / seq->mb_width, col = mb % seq->mb_width;
	predict_plane(cur->y, ref->y, cw, ysize, row, col, 16, mh, mv);
	/* chroma vector: (mv / 2) truncated toward zero, mpeg1.js:562-565 */
	predict_plane(cur->cr, ref->cr, hw, csize, row, col, 8, mh / 2, mv / 2);
	predict_plane(cur->cb, ref->cb, hw, csize, row, col, 8, mh / 2, mv / 2);
}

/* ISO 11172-2 2.4.4.3: a macroblock with both vectors is the average of the two predictions, "//" = rounded
 * to the nearest integer, halves away from zero: (a + b + 1) >> 1 on samples.  `a` holds the forward
 * prediction of the macroblock on entry and the average on exit; `b` the backward prediction. */
static void average_macroblock(const seq_params_t *seq, int cw, int mb, planes_t *a, const planes_t *b) {
	int hw = cw >> 1;
	int row = mb / seq->mb_width, col = mb % seq->mb_width;
	for (int y = 0; y < 16; y++)
		for (int x = 0; x < 16; x++) {
			int i = (row * 16 + y) * cw + col * 16 + x;
			a->y[i] = (uint8_t)((a->y[i] + b->y[i] + 1) >> 1);
		}
	for (int y = 0; y < 8; y++)
		for (int x = 0; x < 8; x++) {
			int i = (row * 8 + y) * hw + col * 8 + x;
			a->cr[i] = (uint8_t)((a->cr[i] + b->cr[i] + 1) >> 1);
			a->cb[i] = (uint8_t)((a->cb[i] + b->cb[i] + 1) >> 1);
		}
}

/* I and P pictures: bwd == NULL, every non-intra macroblock predicts from fwd (mpeg1.js:336-346, 459-687).
 * B pictures (the extension): fwd = the older, bwd = the newer of the two most recent I/P pictures; the record's
 * MBF_MOTION_* bits say which are used. */
static void reconstruct_picture(const seq_params_t *seq, int coded_width, int coded_height,
                                const mb_record_t *hdr, const int16_t *coef,
                                const planes_t *fwd, const planes_t *bwd, planes_t *cur) {
	int cw = coded_width, hw = coded_width >> 1;
	int ysize = coded_width * coded_height, csize = ysize >> 2;
	planes_t tmp = { 0, 0, 0 };
	if (bwd) { tmp.y = (uint8_t *)calloc(ysize, 1); tmp.cr = (uint8_t *)calloc(csize, 1); tmp.cb = (uint8_t *)calloc(csize, 1); }
	for (int mb = 0; mb < seq->mb_size; mb++) {
		const mb_record_t *r = &hdr[mb];
		if (!(r->flags & MBF_PRESENT)) continue; /* untouched: keeps the 2-frames-old content */
		int row = mb / seq->mb_width, col = mb % seq->mb_width;
		bool intra = r->flags & MBF_INTRA;
		if (!intra && !bwd) {
			predict_macroblock(seq, cw, ysize, mb, r->mv_h, r->mv_v, fwd, cur);
		} else if (!intra) {
			int bh = (int16_t)(r->mv_bwd & 0xffffu), bv = (int16_t)(r->mv_bwd >> 16);
			bool use_f = r->flags & MBF_MOTION_FWD, use_b = r->flags & MBF_MOTION_BWD;
			if (use_f || !use_b) predict_macroblock(seq, cw, ysize, mb, r->mv_h, r->mv_v, fwd, cur);
			if (use_b && !use_f) predict_macroblock(seq, cw, ysize, mb, bh, bv, bwd, cur);
			if (use_b && use_f) {
				predict_macroblock(seq, cw, ysize, mb, bh, bv, bwd, &tmp);
				average_macroblock(seq, cw, mb, cur, &tmp);
			}
		}
		for (int block = 0; block < 6; block++) {
			if (!(r->cbp & (0x20 >> block))) continue;
			const int16_t *c = coef + ((size_t)mb * 6 + block) * 64;
			uint8_t *dst; int stride;
			if (block < 4) { /* mpeg1.js:819-828 */
				stride = cw;
				dst = cur->y + (row * 16 + (block & 2 ? 8 : 0)) * cw + col * 16 + (block & 1 ? 8 : 0);
			} else {         /* block 4 -> Cb plane, block 5 -> Cr plane, mpeg1.js:829-834 */
				stride = hw;
				dst = (block == 4 ? cur->cb : cur->cr) + row * 8 * hw + col * 8;
			}
			int px[64];
			if (r->dc_only & (0x20 >> block)) { /* mpeg1.js:838-841, 850-853 */
				int v = (c[0] * ORACLE_PREMULTIPLIER[0] + 128) >> 8;
				for (int k = 0; k < 64; k++) px[k] = v;
			} else {
				for (int k = 0; k < 64; k++) px[k] = c[k] * ORACLE_PREMULTIPLIER[k];
				for (int k = 0; k < 8; k++) idct_pass(px + k, 8, false);
				for (int k = 0; k < 8; k++) idct_pass(px + 8 * k, 1, true);
			}
			for (int y = 0; y < 8; y++)
				for (int x = 0; x < 8; x++) {
					uint8_t *d = dst + y * stride + x;
					*d = clamp255(intra ? px[y * 8 + x] : *d + px[y * 8 + x]); /* mpeg1.js:864-914 */
				}
		}
	}
	if (bwd) free_planes(&tmp);
}

void oracle_reconstruct(const seq_params_t *seq, int coded_width, int coded_height,
                        const mb_record_t *hdr, const int16_t *coef,
                        const planes_t *fwd, planes_t *cur) {
	reconstruct_picture(seq, coded_width, coded_height, hdr, coef, fwd, NULL, cur);
}

/* B picture (extension): see reconstruct_picture */
void oracle_reconstruct_b(const seq_params_t *seq, int coded_width, int coded_height,
                          const mb_record_t *hdr, const int16_t *coef,
                          const planes_t *fwd, const planes_t *bwd, planes_t *cur) {
	reconstruct_picture(seq, coded_width, coded_height, hdr, coef, fwd, bwd, cur);
}

/* ------------------------------------------------------------------------------------------ */
/* The reference's 15-function ABI (src/wasm/mpeg1.h:10-25) on top of the two stages            */

typedef struct mpeg1_decoder_t {
	uint8_t *bytes; uint32_t capacity, length, index; int mode; /* bit buffer, buffer.c */
	bool has_sequence_header;
	float frame_rate;
	int width, height, coded_width, coded_height, coded_size;
	seq_params_t seq;
	planes_t current, forward;
	/* B-picture extension: where B pictures are reconstructed (they are no references) -- two sets written in
	 * turn, like the product's (its copy-out of one B picture overlaps the reconstruction of the next): a
	 * macroblock no slice covers keeps what the B picture before the previous one left there */
	planes_t bout[2];
	int b_cur;
	bool last_was_b;
	mb_record_t *hdr; int16_t *coef;
	picture_info_t last;
} mpeg1_decoder_t;

mpeg1_decoder_t *mpeg1_decoder_create(unsigned int buffer_size, int mode) {
	mpeg1_decoder_t *d = (mpeg1_decoder_t *)calloc(1, sizeof(*d));
	d->bytes = (uint8_t *)malloc(buffer_size ? buffer_size : 1);
	d->capacity = buffer_size; d->mode = mode;
	tries_init();
	return d;
}

void mpeg1_decoder_destroy(mpeg1_decoder_t *d) {
	free(d->bytes);
	if (d->has_sequence_header) { free_planes(&d->current); free_planes(&d->forward); free_planes(&d->bout[0]); free_planes(&d->bout[1]); free(d->hdr); free(d->coef); }
	free(d);
}

/* buffer.c:48-65 get_write_ptr + :167-190 evict + :157-164 resize */
void *mpeg1_decoder_get_write_ptr(mpeg1_decoder_t *d, unsigned int n) {
	uint32_t avail = d->capacity - d->length;
	if (n > avail) {
		if (d->mode == 2) { /* EXPAND */
			uint32_t cap = d->capacity * 2;
			if (cap + avail < n) cap = n - avail;
			d->bytes = (uint8_t *)realloc(d->bytes, cap);
			d->capacity = cap;
			if (d->index > d->length << 3) d->index = d->length << 3;
		} else {            /* EVICT */
			uint32_t pos = d->index >> 3;
			if (pos == d->length || n > avail + pos) { d->length = 0; d->index = 0; }
			else if (pos != 0) {
				memmove(d->bytes, d->bytes + pos, d->length - pos);
				d->length -= pos; d->index -= pos << 3;
			}
		}
	}
	/* buffer.c's sizing can leave less room than it promises (a partly full buffer and a large write: the C build then
	 * writes past its allocation, the JS build throws).  A checker must not corrupt its own heap: make the room. */
	if (d->capacity - d->length < n) {
		d->capacity = d->length + n;
		d->bytes = (uint8_t *)realloc(d->bytes, d->capacity);
	}
	return d->bytes + d->length;
}

int mpeg1_decoder_get_index(mpeg1_decoder_t *d) { return (int)d->index; }
void mpeg1_decoder_set_index(mpeg1_decoder_t *d, unsigned int i) { d->index = i; }

static planes_t alloc_planes(int ysize) {
	planes_t p = { (uint8_t *)calloc(ysize, 1), (uint8_t *)calloc(ysize >> 2, 1), (uint8_t *)calloc(ysize >> 2, 1) };
	return p;
}

/* mpeg1.js:78-153 decodeSequenceHeader + initBuffers */
static void parse_sequence_header(mpeg1_decoder_t *d, bits_t *b) {
	d->width = bits_read(b, 12);
	d->height = bits_read(b, 12);
	bits_skip(b, 4);
	d->frame_rate = ORACLE_PICTURE_RATE[bits_read(b, 4)];
	bits_skip(b, 18 + 1 + 10 + 1);
	if (bits_read(b, 1)) { for (int i = 0; i < 64; i++) d->seq.intra_q[ORACLE_ZIG_ZAG[i]] = (uint8_t)bits_read(b, 8); }
	else memcpy(d->seq.intra_q, ORACLE_DEFAULT_INTRA_QUANT, 64);
	if (bits_read(b, 1)) { for (int i = 0; i < 64; i++) d->seq.non_intra_q[ORACLE_ZIG_ZAG[i]] = (uint8_t)bits_read(b, 8); }
	else memset(d->seq.non_intra_q, 16, 64);
	int mbw = (d->width + 15) >> 4, mbh = (d->height + 15) >> 4;
	d->seq.mb_width = mbw; d->seq.mb_size = mbw * mbh;
	d->coded_width = mbw << 4; d->coded_height = mbh << 4;
	d->coded_size = d->coded_width * d->coded_height;
	d->current = alloc_planes(d->coded_size);
	d->forward = alloc_planes(d->coded_size);
	d->bout[0] = alloc_planes(d->coded_size);
	d->bout[1] = alloc_planes(d->coded_size);
	d->hdr = (mb_record_t *)calloc(d->seq.mb_size, sizeof(mb_record_t));
	d->coef = (int16_t *)calloc((size_t)d->seq.mb_size * MB_COEF_INT16, sizeof(int16_t));
	d->has_sequence_header = true;
}

/* mpeg1.c:812-819 */
void mpeg1_decoder_did_write(mpeg1_decoder_t *d, unsigned int n) {
	d->length += n;
	if (!d->has_sequence_header) {
		bits_t b = { d->bytes, d->length, d->index };
		if (bits_find_start_code(&b, 0xB3) != -1) parse_sequence_header(d, &b);
		d->index = b.index;
	}
}

int mpeg1_decoder_has_sequence_header(mpeg1_decoder_t *d) { return d->has_sequence_header; }
float mpeg1_decoder_get_frame_rate(mpeg1_decoder_t *d) { return d->frame_rate; }
int mpeg1_decoder_get_coded_size(mpeg1_decoder_t *d) { return d->coded_size; }
int mpeg1_decoder_get_width(mpeg1_decoder_t *d) { return d->width; }
int mpeg1_decoder_get_height(mpeg1_decoder_t *d) { return d->height; }
/* most recently decoded picture = forward after the swap (mpeg1.c:841-851, SURVEY Q17) */
void *mpeg1_decoder_get_y_ptr(mpeg1_decoder_t *d) { return d->last_was_b ? d->bout[d->b_cur ^ 1].y : d->forward.y; }
void *mpeg1_decoder_get_cr_ptr(mpeg1_decoder_t *d) { return d->last_was_b ? d->bout[d->b_cur ^ 1].cr : d->forward.cr; }
void *mpeg1_decoder_get_cb_ptr(mpeg1_decoder_t *d) { return d->last_was_b ? d->bout[d->b_cur ^ 1].cb : d->forward.cb; }

/* mpeg1.c:853-864 + decode_picture :947-995 */
bool mpeg1_decoder_decode(mpeg1_decoder_t *d) {
	if (!d->has_sequence_header) return false;
	bits_t b = { d->bytes, d->length, d->index };
	int found = bits_find_start_code(&b, 0x00);
	d->index = b.index;
	if (found == -1) return false;
	memset(d->hdr, 0, (size_t)d->seq.mb_size * sizeof(mb_record_t));
	oracle_parse_picture(d->bytes, d->length, d->index, &d->seq, &d->last, d->hdr, d->coef);
	d->index = d->last.end_bit;
	if (d->last.status == PIC_DECODED && d->last.picture_type == 3) {
		/* extension: after the swaps `current` holds the older and `forward` the newer of the two most recent
		 * I/P pictures = the B picture's forward (past) and backward (future) reference.  Pictures leave in
		 * CODED order; no swap, a B picture is never a reference. */
		oracle_reconstruct_b(&d->seq, d->coded_width, d->coded_height, d->hdr, d->coef, &d->current, &d->forward, &d->bout[d->b_cur]);
		d->b_cur ^= 1;
		d->last_was_b = true;
	} else if (d->last.status == PIC_DECODED) {
		oracle_reconstruct(&d->seq, d->coded_width, d->coded_height, d->hdr, d->coef, &d->forward, &d->current);
		planes_t t = d->forward; d->forward = d->current; d->current = t;
		d->last_was_b = false;
	}
	return true;
}

/* The product's two extension entry points under the same names (include/jsmpeg_b200.h), so that the shared host
 * class (jsmpeg_b200/decoder.py) drives this checker exactly like the product.  "decode_b" is process-wide here. */
int jsmpeg_b200_decoder_set_option(mpeg1_decoder_t *d, const char *name, int value) {
	(void)d;
	if (strcmp(name, "decode_b") == 0) { g_decode_b = value; return 0; }
	return -1;
}
int jsmpeg_b200_decoder_last_picture(mpeg1_decoder_t *d, int *picture_type, int *temporal_reference) {
	if (!d->last.picture_type) return -1;
	if (picture_type) *picture_type = d->last.picture_type;
	if (temporal_reference) { /* 10 bits right after the picture start code */
		uint32_t p = d->last.start_byte;
		*temporal_reference = p + 1 < d->length ? (d->bytes[p] << 2 | d->bytes[p + 1] >> 6) : 0;
	}
	return 0;
}

/* test hooks */
void oracle_idct(int *block) { /* the 2-D transform alone, for unit parity against the reference's idct() */
	for (int k = 0; k < 8; k++) idct_pass(block + k, 8, false);
	for (int k = 0; k < 8; k++) idct_pass(block + 8 * k, 1, true);
}
const picture_info_t *oracle_last_picture_info(mpeg1_decoder_t *d) { return &d->last; }
const mb_record_t *oracle_last_mb_records(mpeg1_decoder_t *d) { return d->hdr; }
const int16_t *oracle_last_coefficients(mpeg1_decoder_t *d) { return d->coef; }
const seq_params_t *oracle_seq_params(mpeg1_decoder_t *d) { return &d->seq; }

/* FNV-1a 64 continuation over caller memory: the picture hash that bench.py and the tests compare decoded planes
 * by (the hash is serial; in Python it would take seconds per picture) */
uint64_t oracle_hash_bytes(uint64_t h, const uint8_t *p, size_t n) {
	for (size_t i = 0; i < n; i++) { h ^= p[i]; h *= 1099511628211ULL; }
	return h;
}

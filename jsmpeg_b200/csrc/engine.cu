// engine.cu -- host side of libjsmpeg_b200.so: stream state, HBM residency, wave planning, and
// the two C ABIs declared in include/jsmpeg_b200.h.
//
// What stays on the host is exactly what is bookkeeping in the reference too: the bit-buffer write
// protocol (src/wasm/buffer.c:48-71, 157-190; bitbuffer.h), the sequence header (src/mpeg1.js:78-153,
// parsed once per stream) and the decode() state machine (src/wasm/mpeg1.c:853-864, 947-995: which
// picture is next, where the bit index ends up, when planes swap).  All per-byte, per-bit and
// per-pixel work runs in the kernels (scan.cu, parse.cu, recon.cu).  There is no CPU fallback:
// without a usable CUDA device a decoder is created DEAD -- every entry point returns its failure
// value (decode() == false, like "no sequence header yet"), the reason is printed once and kept for
// jsmpeg_b200_batch_last_error.  Nothing here calls abort(): a plugin must not take its host process
// (a Node player) down.
//
// Wave model.  decode() on a stream needs (a) the next picture start code, (b) that picture's
// records, (c) its reconstruction from the previous picture.  (a) comes from the start-code index
// built when bytes become resident; (b) for MANY pictures (all streams x pictures ahead) is one
// parse wave, one warp per picture; (c) is one launch per picture STEP covering every stream
// that has a picture at that step.  The reference's serial semantics are re-established on the
// host after the parse: picture j+1 of a stream is accepted only if its start code is the first
// one at/after the bit index where picture j's parse ended (otherwise the look-ahead is discarded
// and re-planned from there).
//
// Pipeline.  A round's parse wave can be cut into CHUNKS by picture ordinal (pictures [kG, (k+1)G)
// of every stream; option "chunk_pictures"); all chunks are queued on the parse stream at once, each
// followed by the read-back of its picture infos.  The host then takes chunk after chunk: waits for
// that chunk's infos only, does the acceptance above, and queues the chunk's reconstruct launches on
// a SECOND stream -- while the parse of the following chunks is running.  Stage 1 (latency-bound, few
// resident warps) and stage 2 (bandwidth / issue-bound) are natural co-runners; round 1 serialised
// them with a host synchronisation between the parse wave and the first reconstruct launch.
#include <sched.h>

#include <algorithm>
#include <cstring>
#include <deque>
#include <string>
#include <vector>

#include "bitbuffer.h"
#include "common.cuh"
#include "../../include/jsmpeg_b200.h"

namespace {

constexpr int HOST_RING = 4;
constexpr uint32_t ES_PAD = 512;  // readable, zeroed slack after the ES mirror (the walk's ring prefetches 64 bytes ahead)

template <typename T>
T *dev_alloc(size_t n) {
	T *p = nullptr;
	CUDA_CHECK(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
	return p;
}
template <typename T>
T *pinned_alloc(size_t n) {
	T *p = nullptr;
	CUDA_CHECK(cudaHostAlloc(&p, std::max<size_t>(n, 1) * sizeof(T), cudaHostAllocDefault));
	return p;
}

// the bit buffer lives in pinned host memory (H2D copies of new bytes run at PCIe speed)
void *bb_pinned_alloc(size_t n, void *) { return pinned_alloc<uint8_t>(n); }
void bb_pinned_release(void *p, void *) { (void)cudaFreeHost(p); }
const bitbuffer::Allocator kPinned = {bb_pinned_alloc, bb_pinned_release, nullptr};

struct Parsed {
	uint32_t pos;           // byte position of the 00 00 01 00 start code
	uint32_t len_at_parse;  // buffer length the parse saw
	int slot;
	bool ready;             // `info` has arrived from the device
	picture_info_t info;
};

struct Stream {
	bitbuffer::Buffer bb;  // host bit buffer (pinned) -- src/wasm/buffer.c
	// sequence header
	bool has_seq = false;
	float frame_rate = 0.f;
	int width = 0, height = 0, coded_size = 0;
	uint32_t seq_end_index = 0;  // bit index right after the sequence header
	SeqParams seq{};
	SeqParams *d_seq = nullptr;
	// ES mirror in HBM + start-code index
	uint8_t *d_es = nullptr;
	uint32_t d_capacity = 0, d_valid = 0;
	std::vector<uint32_t> pics;  // sorted byte positions of picture start codes (00 00 01 00)
	std::vector<uint32_t> codes, pic_code;  // every start-code prefix (00 00 01), sorted; pics[k] == codes[pic_code[k]]
	uint32_t codes_classified = 0;          // codes[0 .. codes_classified) have had their fourth byte looked at
	uint32_t scanned = 0;        // every prefix with pos + 2 < scanned is in `codes`
	uint32_t scan_from = 0;      // the span a pending scan covers starts here
	bool scan_pending = false;
	// planes: two sets in HBM (ping-pong like mpeg1.js:221-246), a host ring for OUT_HOST
	uint8_t *d_planes[2] = {nullptr, nullptr};
	int cur = 0;  // set written by the next I/P picture; forward = 1 - cur
	uint8_t *h_planes[HOST_RING] = {};
	int h_head = -1;
	// B-picture extension ("decode_b"): two more sets in HBM, written in turn -- a B picture is no reference, the
	// ping-pong above is untouched by it; d_last = the set holding the most recently decoded picture
	uint8_t *d_planes_b[2] = {nullptr, nullptr};
	int b_cur = 0;
	uint8_t *d_last = nullptr;
	int last_type = 0, last_temporal = 0;  // picture_coding_type / temporal_reference of the last picture decode() consumed
	uint8_t *d_rgba = nullptr;
	std::vector<int16_t> ts_bound;     // device TS demux: the stream id every PID is bound to, 0 = none (ts.js pidsToStreamIds)
	std::vector<uint8_t> ts_leftover;  // ... and the bytes the last write_ts left over (ts.js leftoverBytes)
	// parsed-ahead pictures, consecutive, front = next picture decode() consumes
	std::deque<Parsed> cache;
};

}  // namespace

struct jsmpeg_b200_batch_t {
	int device = 0;
	bool dead = false;  // a CUDA call failed: every entry point returns its failure value from now on
	std::string error;
	std::vector<uint8_t> dead_scratch;  // where get_write_ptr points a caller's memcpy once dead
	std::vector<Stream> streams;
	// start-code scan of all streams in one launch (scan.cu): span list, per-span hit counts and positions;
	// and the device's copy of every stream's sorted prefix list (ParseTask::codes), one row per stream
	ScanSpan *d_spans = nullptr, *h_spans = nullptr;
	uint32_t *d_scan_counts = nullptr, *h_scan_counts = nullptr, *d_scan_pos = nullptr, *h_scan_pos = nullptr;
	uint32_t scan_rows = 0, scan_seg = 0;       // room: spans, positions per span
	uint32_t *d_codes = nullptr, *h_codes = nullptr;
	uint32_t codes_rows = 0, codes_stride = 0;  // rows = streams, stride = entries per row
	cudaStream_t st_main = nullptr, st_recon = nullptr, st_copy = nullptr;  // uploads + scan + parse | reconstruct | copy-out
	cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_mid = nullptr, ev_step = nullptr, ev_round = nullptr, ev_copied[2] = {nullptr, nullptr};
	std::vector<cudaEvent_t> ev_info;            // per chunk: its picture infos are on the host
	std::vector<cudaEvent_t> ev_rec0, ev_rec1;   // per chunk: around its reconstruct launches (timing)
	// record slots
	unsigned max_slots_req = 0;
	int slot_mb = 0, n_slots = 0;
	mb_record_t *d_hdr = nullptr;
	int16_t *d_coef = nullptr;
	uint2 *d_park = nullptr;
	uint4 *d_stage = nullptr;  // per slot: stage_entries_for(slot_mb) x 64 B (lane-parallel walk, relative records)
	picture_info_t *d_info = nullptr, *h_info = nullptr;
	std::vector<int> free_slots;
	int lookahead = 1;
	bool decode_b = false;       // the B-picture extension: off = B pictures are skipped like the reference does (mpeg1.js:181-184)
	bool slice_walk = false;     // I/P pictures of >= SLICE_WALK_MIN_SLICES slices go to the one-lane-per-slice walk (walk_slices.cuh)
	int chunk_pictures = 0;      // G of the pipeline; 0 = the whole wave is one chunk
	int chunk_min_wave = 256;    // waves with fewer new pictures stay whole
	int chunk_streams = 3;       // chunks are parsed on this many streams in turn (1 = on the main stream, forked into size groups)
	// pictures with a walk kernel of their own (B pictures; with "slice_walk", I/P pictures of many slices) are
	// walked beside the others, on these streams
	cudaStream_t st_side[2] = {nullptr, nullptr};
	cudaEvent_t ev_sfork = nullptr, ev_sjoin[2] = {nullptr, nullptr};
	cudaStream_t st_chunk[4] = {nullptr, nullptr, nullptr, nullptr};
	cudaEvent_t ev_fed = nullptr, ev_chunk_done[4] = {nullptr, nullptr, nullptr, nullptr};
	bool recon_pending = false;  // reconstruct launches of an earlier round may still read record slots
	// task staging
	ParseTask *h_ptasks = nullptr, *d_ptasks = nullptr;
	int ptask_cap = 0;
	ReconTask *h_rtasks = nullptr, *d_rtasks = nullptr;
	int rtask_cap = 0;
	uint64_t copy_steps = 0;  // reconstruct launches with a copy-out so far (event parity)
	ParseFork fork{};
	std::vector<void *> copy_dst, copy_src;
	std::vector<size_t> copy_size;
	bool batch_copy_ok = true;
	TsScratch *ts = nullptr;
	jsmpeg_b200_stats_t stats{};
};

namespace {

using Batch = jsmpeg_b200_batch_t;

void use_device(Batch *b) { CUDA_CHECK(cudaSetDevice(b->device)); }

void mark_dead(Batch *b, const char *what) {
	if (!b->dead) fprintf(stderr, "%s\njsmpeg_b200: decoder disabled (decode() returns false from now on)\n", what);
	b->dead = true;
	if (b->error.empty()) b->error = what;
}

// Every C-ABI entry point that touches CUDA runs through here.
template <typename R, typename F>
R guarded(Batch *b, R fail, F &&f) {
	if (!b || b->dead) return fail;
	try {
		return f();
	} catch (const std::exception &e) {
		mark_dead(b, e.what());
	} catch (...) {
		mark_dead(b, "jsmpeg_b200: unknown failure");
	}
	return fail;
}
template <typename F>
void guarded_void(Batch *b, F &&f) {
	guarded<int>(b, 0, [&] { f(); return 0; });
}

void release_slot(Batch *b, int slot) { b->free_slots.push_back(slot); }

void flush_cache(Batch *b, Stream &s) {
	for (auto &p : s.cache) release_slot(b, p.slot);
	s.cache.clear();
}

void forget_index(Batch *b, Stream &s) {
	flush_cache(b, s);
	s.pics.clear();
	s.codes.clear();
	s.pic_code.clear();
	s.codes_classified = 0;
	s.scanned = 0;
	s.d_valid = 0;
}

// ---- bit buffer (host) ------------------------------------------------------------------------

// src/wasm/buffer.c:48-65 get_write_ptr, :167-190 evict (bitbuffer.h)
void *stream_get_write_ptr(Batch *b, Stream &s, uint32_t n) {
	bool moved = false;
	uint8_t *p = bitbuffer::get_write_ptr(s.bb, n, kPinned, moved);
	if (moved) forget_index(b, s);  // byte positions changed: the HBM mirror, the index and the look-ahead are void
	if (!p) throw std::runtime_error("jsmpeg_b200: bit buffer cannot hold the write (more than 4 GiB - 1 bytes)");
	return p;
}

// MSB-first reader for the (tiny, once-per-stream) sequence header on the host
struct HostBits {
	const uint8_t *p;
	uint32_t len, idx;
	uint32_t read(int n) {
		uint32_t v = 0;
		for (int i = 0; i < n; i++, idx++) {
			uint32_t byte = idx >> 3;
			v = (v << 1) | (byte < len ? (p[byte] >> (7 - (idx & 7))) & 1u : 0u);
		}
		return v;
	}
};

const float kPictureRate[16] = {0.f, 23.976f, 24.f, 25.f, 29.97f, 30.f, 50.f, 59.94f, 60.f, 0, 0, 0, 0, 0, 0, 0};
const uint8_t kZigZag[64] = {0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48,
                             41, 34, 27, 20, 13, 6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22,
                             15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
const uint8_t kDefaultIntraQ[64] = {8, 16, 19, 22, 26, 27, 29, 34, 16, 16, 22, 24, 27, 29, 34, 37,
                                    19, 22, 26, 27, 29, 34, 34, 38, 22, 22, 26, 27, 29, 34, 37, 40,
                                    22, 26, 27, 29, 32, 35, 40, 48, 26, 27, 29, 32, 35, 40, 48, 58,
                                    26, 27, 29, 34, 38, 46, 56, 69, 27, 29, 35, 38, 46, 56, 69, 83};

// src/mpeg1.js:78-153 decodeSequenceHeader + initBuffers (first header only, mpeg1.c:812-819)
void parse_sequence_header(Batch *b, Stream &s, uint32_t bit_index) {
	HostBits hb{s.bb.bytes, s.bb.length, bit_index};
	s.width = (int)hb.read(12);
	s.height = (int)hb.read(12);
	hb.read(4);
	s.frame_rate = kPictureRate[hb.read(4)];
	hb.read(18 + 1 + 10 + 1);
	if (hb.read(1)) { for (int i = 0; i < 64; i++) s.seq.intra_q[kZigZag[i]] = (uint8_t)hb.read(8); }
	else memcpy(s.seq.intra_q, kDefaultIntraQ, 64);
	if (hb.read(1)) { for (int i = 0; i < 64; i++) s.seq.non_intra_q[kZigZag[i]] = (uint8_t)hb.read(8); }
	else memset(s.seq.non_intra_q, 16, 64);
	seq_fill_xq(s.seq);
	s.bb.index = hb.idx;
	s.seq_end_index = hb.idx;
	s.seq.mb_width = (s.width + 15) >> 4;
	s.seq.mb_height = (s.height + 15) >> 4;
	s.seq.mb_size = s.seq.mb_width * s.seq.mb_height;
	s.seq.coded_width = s.seq.mb_width << 4;
	s.seq.coded_height = s.seq.mb_height << 4;
	s.coded_size = s.seq.coded_width * s.seq.coded_height;
	s.has_seq = true;

	const size_t plane_bytes = (size_t)s.coded_size * 3 / 2;
	s.d_seq = dev_alloc<SeqParams>(1);
	CUDA_CHECK(cudaMemcpyAsync(s.d_seq, &s.seq, sizeof(SeqParams), cudaMemcpyHostToDevice, b->st_main));
	for (int i = 0; i < 2; i++) {
		// + coded_width + 64: stage 2's row loads may touch (never use) up to one row past a plane set's end
		s.d_planes[i] = dev_alloc<uint8_t>(plane_bytes + s.seq.coded_width + 64);
		CUDA_CHECK(cudaMemsetAsync(s.d_planes[i], 0, plane_bytes + s.seq.coded_width + 64, b->st_main));  // JS typed arrays start zeroed
	}
	for (int i = 0; i < HOST_RING; i++) {
		s.h_planes[i] = pinned_alloc<uint8_t>(plane_bytes);
		memset(s.h_planes[i], 0, plane_bytes);
	}
	CUDA_CHECK(cudaStreamSynchronize(b->st_main));  // s.seq is read by the async copy
}

// src/wasm/mpeg1.c:812-819 did_write
void stream_did_write(Batch *b, Stream &s, uint32_t n) {
	if ((uint64_t)s.bb.length + n > s.bb.capacity) n = s.bb.capacity - s.bb.length;  // never beyond what get_write_ptr handed out
	s.bb.length += n;
	if (!s.has_seq) {
		// findStartCode(SEQUENCE): serial host scan of the not-yet-consumed head of the stream
		uint32_t i = (s.bb.index + 7) >> 3;
		bool found = false;
		for (; i + 3 < s.bb.length; i++) {
			if (s.bb.bytes[i] == 0 && s.bb.bytes[i + 1] == 0 && s.bb.bytes[i + 2] == 1) {
				if (s.bb.bytes[i + 3] == 0xB3) { found = true; break; }
				i += 3;  // index jumps past the code (buffer.js:121-123)
			}
		}
		if (found) parse_sequence_header(b, s, (i + 4) << 3);
		else s.bb.index = s.bb.length << 3;
	}
}

// ---- residency: H2D of new bytes + start-code scan -----------------------------------------------

// Room for `need` ES bytes (+ pad) in the HBM mirror; what is already resident stays resident.
void reserve_device_es(Batch *b, Stream &s, uint32_t need) {
	if ((uint64_t)need + ES_PAD <= s.d_capacity) return;
	uint64_t cap = std::max<uint64_t>((uint64_t)need + ES_PAD, (uint64_t)s.d_capacity * 2);
	cap = std::min<uint64_t>((cap + 255u) & ~255ull, 0xffffff00ull);
	uint8_t *n = dev_alloc<uint8_t>(cap);
	if (s.d_es) {
		if (s.d_valid) CUDA_CHECK(cudaMemcpyAsync(n, s.d_es, s.d_valid, cudaMemcpyDeviceToDevice, b->st_main));
		CUDA_CHECK(cudaStreamSynchronize(b->st_main));
		CUDA_CHECK(cudaFree(s.d_es));
	}
	s.d_es = n;
	s.d_capacity = (uint32_t)cap;
}

// Room for `rows` spans with `seg` positions each (contents are per scan: nothing to keep).
void reserve_scan(Batch *b, uint32_t rows, uint32_t seg) {
	if (rows <= b->scan_rows && seg <= b->scan_seg) return;
	rows = std::max(rows, b->scan_rows);
	seg = std::max(seg, b->scan_seg);
	if (b->d_spans) CUDA_CHECK(cudaFree(b->d_spans));
	if (b->d_scan_counts) CUDA_CHECK(cudaFree(b->d_scan_counts));
	if (b->d_scan_pos) CUDA_CHECK(cudaFree(b->d_scan_pos));
	if (b->h_spans) CUDA_CHECK(cudaFreeHost(b->h_spans));
	if (b->h_scan_counts) CUDA_CHECK(cudaFreeHost(b->h_scan_counts));
	if (b->h_scan_pos) CUDA_CHECK(cudaFreeHost(b->h_scan_pos));
	b->d_spans = nullptr; b->d_scan_counts = nullptr; b->d_scan_pos = nullptr;
	b->h_spans = nullptr; b->h_scan_counts = nullptr; b->h_scan_pos = nullptr;
	b->scan_rows = b->scan_seg = 0;
	b->d_spans = dev_alloc<ScanSpan>(rows);
	b->h_spans = pinned_alloc<ScanSpan>(rows);
	b->d_scan_counts = dev_alloc<uint32_t>(rows);
	b->h_scan_counts = pinned_alloc<uint32_t>(rows);
	b->d_scan_pos = dev_alloc<uint32_t>((size_t)rows * seg);
	b->h_scan_pos = pinned_alloc<uint32_t>((size_t)rows * seg);
	b->scan_rows = rows;
	b->scan_seg = seg;
}

// One launch over the pending spans (h_spans[0 .. n)); the counts come back to h_scan_counts.
void launch_scan(Batch *b, int n, uint32_t longest) {
	CUDA_CHECK(cudaMemcpyAsync(b->d_spans, b->h_spans, n * sizeof(ScanSpan), cudaMemcpyHostToDevice, b->st_main));
	CUDA_CHECK(cudaMemsetAsync(b->d_scan_counts, 0, n * sizeof(uint32_t), b->st_main));
	launch_scan_start_codes(b->d_spans, n, longest, b->d_scan_pos, b->scan_seg, b->d_scan_counts, b->st_main);
	b->stats.kernel_launches++;
	CUDA_CHECK(cudaMemcpyAsync(b->h_scan_counts, b->d_scan_counts, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, b->st_main));
}

// The device's copy of every stream's prefix list: row si = streams[si].codes.  The host has them all, so a
// change of geometry (more streams, a longer list) just stages everything again.  Returns true if rebuilt.
bool reserve_codes(Batch *b, uint32_t rows, uint32_t entries) {
	if (rows == b->codes_rows && entries <= b->codes_stride) return false;
	const uint32_t stride = std::max<uint32_t>(std::max<uint32_t>(2 * b->codes_stride, entries + 256u), 1024u);
	if (b->d_codes) {
		CUDA_CHECK(cudaStreamSynchronize(b->st_main));  // (tasks of an earlier round may still name the old rows)
		CUDA_CHECK(cudaStreamSynchronize(b->st_recon));
		CUDA_CHECK(cudaFree(b->d_codes));
	}
	if (b->h_codes) CUDA_CHECK(cudaFreeHost(b->h_codes));
	b->d_codes = nullptr; b->h_codes = nullptr;
	b->codes_rows = b->codes_stride = 0;
	b->d_codes = dev_alloc<uint32_t>((size_t)rows * stride);
	b->h_codes = pinned_alloc<uint32_t>((size_t)rows * stride);
	b->codes_rows = rows;
	b->codes_stride = stride;
	return true;
}

void begin_upload(Batch *b, Stream &s) {
	s.scan_pending = false;
	if (s.d_valid >= s.bb.length && s.scanned >= s.bb.length) return;
	reserve_device_es(b, s, s.bb.length);
	if (s.d_valid < s.bb.length) {
		uint32_t from = s.d_valid & ~15u;
		CUDA_CHECK(cudaMemcpyAsync(s.d_es + from, s.bb.bytes + from, s.bb.length - from, cudaMemcpyHostToDevice, b->st_main));
		b->stats.h2d_bytes += s.bb.length - from;
		s.d_valid = s.bb.length;
		// the kernels rely on zeros right after the data (bytes past the end read as 0, like JS)
		CUDA_CHECK(cudaMemsetAsync(s.d_es + s.bb.length, 0, ES_PAD, b->st_main));
	}
	if (s.scanned < s.bb.length) {
		s.scan_from = s.scanned >= 2 ? s.scanned - 2 : 0;  // a prefix needs its three bytes: those from scanned - 2 on were not complete
		s.scan_pending = true;  // (upload_all scans all pending spans in one launch)
	}
}

long upload_all(Batch *b) {
	CUDA_CHECK(cudaEventRecord(b->ev_a, b->st_main));
	const int S = (int)b->streams.size();
	std::vector<int> pending;
	uint32_t longest = 0, seg = 4096u;
	for (int si = 0; si < S; si++) {
		Stream &s = b->streams[si];
		begin_upload(b, s);
		if (!s.scan_pending) continue;
		pending.push_back(si);
		const uint32_t span = s.bb.length - (s.scan_from & ~15u);
		longest = std::max(longest, span);
		// room for one start code per 512 bytes (FFmpeg streams: two per picture of tens of KiB; a slice per
		// macroblock row: ~70 per picture).  A stream that packs them denser overflows its list; the scan is
		// then repeated with the count it reported.
		seg = std::max(seg, span / 512u + 16u);
	}
	if (!pending.empty()) {
		const int n = (int)pending.size();
		reserve_scan(b, (uint32_t)n, seg);
		for (int k = 0; k < n; k++) {
			const Stream &s = b->streams[pending[k]];
			b->h_spans[k] = ScanSpan{s.d_es, s.scan_from, s.bb.length};
		}
		launch_scan(b, n, longest);
		CUDA_CHECK(cudaEventRecord(b->ev_b, b->st_main));
		CUDA_CHECK(cudaStreamSynchronize(b->st_main));
		float ms = 0;
		CUDA_CHECK(cudaEventElapsedTime(&ms, b->ev_a, b->ev_b));
		b->stats.scan_ms += ms;
		uint32_t most = *std::max_element(b->h_scan_counts, b->h_scan_counts + n);
		if (most > b->scan_seg) {
			// a list overflowed (hostile input: start codes cannot overlap, so at most length / 3 of them): once
			// more, with room for the count the kernel reported
			reserve_scan(b, (uint32_t)n, most + 16u);
			for (int k = 0; k < n; k++) {  // (the pinned span list was reallocated)
				const Stream &s = b->streams[pending[k]];
				b->h_spans[k] = ScanSpan{s.d_es, s.scan_from, s.bb.length};
			}
			launch_scan(b, n, longest);
			CUDA_CHECK(cudaStreamSynchronize(b->st_main));
			most = *std::max_element(b->h_scan_counts, b->h_scan_counts + n);
			if (most > b->scan_seg) throw std::runtime_error("jsmpeg_b200: start-code index overflow after a rescan");
		}
		if (most) {  // the positions of all spans in one (strided) copy
			CUDA_CHECK(cudaMemcpy2DAsync(b->h_scan_pos, (size_t)b->scan_seg * sizeof(uint32_t), b->d_scan_pos,
			                             (size_t)b->scan_seg * sizeof(uint32_t), (size_t)most * sizeof(uint32_t), (size_t)n,
			                             cudaMemcpyDeviceToHost, b->st_main));
			b->stats.d2h_bytes += (uint64_t)most * n * sizeof(uint32_t);
			CUDA_CHECK(cudaStreamSynchronize(b->st_main));
		}
		bool grew = false;
		for (int k = 0; k < n; k++) {
			Stream &s = b->streams[pending[k]];
			uint32_t *hits = b->h_scan_pos + (size_t)k * b->scan_seg;
			const uint32_t cnt = b->h_scan_counts[k];
			std::sort(hits, hits + cnt);
			// the rescanned window starts 2 bytes before the old frontier, so nothing is reported twice
			s.codes.insert(s.codes.end(), hits, hits + cnt);
			grew |= cnt != 0;
			s.scanned = s.bb.length;
			s.scan_pending = false;
		}
		if (grew) {  // the device's copy, for the lane-parallel walk's slice ends: every row that changed, in one copy
			size_t longest_list = 0;
			for (auto &s : b->streams) longest_list = std::max(longest_list, s.codes.size());
			const bool rebuilt = reserve_codes(b, (uint32_t)S, (uint32_t)longest_list);
			for (int si = 0; si < S; si++) {
				const Stream &s = b->streams[si];
				// (a rewound stream's list starts over: staging whole rows keeps this free of bookkeeping; they are short)
				if (!s.codes.empty() && (rebuilt || std::find(pending.begin(), pending.end(), si) != pending.end()))
					memcpy(b->h_codes + (size_t)si * b->codes_stride, s.codes.data(), s.codes.size() * sizeof(uint32_t));
			}
			CUDA_CHECK(cudaMemcpy2DAsync(b->d_codes, (size_t)b->codes_stride * sizeof(uint32_t), b->h_codes,
			                             (size_t)b->codes_stride * sizeof(uint32_t), longest_list * sizeof(uint32_t), (size_t)S,
			                             cudaMemcpyHostToDevice, b->st_main));
			b->stats.h2d_bytes += (uint64_t)longest_list * S * sizeof(uint32_t);
			CUDA_CHECK(cudaStreamSynchronize(b->st_main));  // the pinned staging is written again by the next scan
		}
	}
	// picture start codes = prefixes whose fourth byte is 00 and inside the buffer (findStartCode, buffer.js:130-139).
	// Only the very last prefix can still be waiting for its fourth byte.
	long total = 0;
	for (auto &s : b->streams) {
		while (s.codes_classified < s.codes.size()) {
			const uint32_t p = s.codes[s.codes_classified];
			if (p + 3u >= s.bb.length) break;
			if (s.bb.bytes[p + 3u] == 0) { s.pics.push_back(p); s.pic_code.push_back(s.codes_classified); }
			s.codes_classified++;
		}
		total += (long)s.pics.size();
	}
	return total;
}

// ---- record slots ----------------------------------------------------------------------------------

void ensure_pool(Batch *b) {
	int need_mb = 0;
	for (auto &s : b->streams) if (s.has_seq) need_mb = std::max(need_mb, s.seq.mb_size);
	if (need_mb <= b->slot_mb || need_mb == 0) return;
	for (auto &s : b->streams) flush_cache(b, s);
	CUDA_CHECK(cudaStreamSynchronize(b->st_main));
	CUDA_CHECK(cudaStreamSynchronize(b->st_recon));
	b->recon_pending = false;
	if (b->d_hdr) { CUDA_CHECK(cudaFree(b->d_hdr)); b->d_hdr = nullptr; }
	if (b->d_coef) { CUDA_CHECK(cudaFree(b->d_coef)); b->d_coef = nullptr; }
	if (b->d_park) { CUDA_CHECK(cudaFree(b->d_park)); b->d_park = nullptr; }
	if (b->d_stage) { CUDA_CHECK(cudaFree(b->d_stage)); b->d_stage = nullptr; }
	if (b->d_info) { CUDA_CHECK(cudaFree(b->d_info)); b->d_info = nullptr; }
	if (b->h_info) { CUDA_CHECK(cudaFreeHost(b->h_info)); b->h_info = nullptr; }
	b->slot_mb = 0;
	b->n_slots = 0;
	b->free_slots.clear();
	// per macroblock: 16 B record + 6 x 128 B coefficient blocks + 6 x 8 B {bit offset, dc} side array; per picture
	// the lane-parallel walk's staging entries
	const size_t slot_bytes = (size_t)need_mb * (sizeof(mb_record_t) + MB_COEF_INT16 * sizeof(int16_t) + 6 * sizeof(uint2)) +
	                          (size_t)stage_entries_for(need_mb) * 64;
	size_t n = b->max_slots_req;
	size_t free_b = 0, total_b = 0;
	CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
	const size_t fit = (size_t)(0.9 * (double)free_b) / slot_bytes;  // a request beyond the device is cut, not fatal
	if (n == 0) n = std::min<size_t>((size_t)(0.45 * (double)free_b) / slot_bytes, 4096);
	n = std::max<size_t>(std::min(n, fit), 2);
	b->d_hdr = dev_alloc<mb_record_t>(n * need_mb);
	b->d_coef = dev_alloc<int16_t>(n * need_mb * MB_COEF_INT16);
	b->d_park = dev_alloc<uint2>(n * need_mb * 6);
	b->d_stage = dev_alloc<uint4>(n * (size_t)stage_entries_for(need_mb) * 4);
	b->d_info = dev_alloc<picture_info_t>(n);
	b->h_info = pinned_alloc<picture_info_t>(n);
	b->slot_mb = need_mb;
	b->n_slots = (int)n;
	for (int i = (int)n - 1; i >= 0; i--) b->free_slots.push_back(i);
}

void ensure_task_caps(Batch *b, int n_parse, int n_recon) {
	if (n_parse > b->ptask_cap) {
		if (b->h_ptasks) { CUDA_CHECK(cudaFreeHost(b->h_ptasks)); b->h_ptasks = nullptr; }
		if (b->d_ptasks) { CUDA_CHECK(cudaFree(b->d_ptasks)); b->d_ptasks = nullptr; }
		const int cap = std::max(n_parse, b->ptask_cap * 2);
		b->ptask_cap = 0;
		b->h_ptasks = pinned_alloc<ParseTask>(cap);
		b->d_ptasks = dev_alloc<ParseTask>(cap);
		b->ptask_cap = cap;
	}
	if (n_recon > b->rtask_cap) {
		if (b->h_rtasks) { CUDA_CHECK(cudaFreeHost(b->h_rtasks)); b->h_rtasks = nullptr; }
		if (b->d_rtasks) { CUDA_CHECK(cudaFree(b->d_rtasks)); b->d_rtasks = nullptr; }
		const int cap = std::max(n_recon, b->rtask_cap * 2);
		b->rtask_cap = 0;
		b->h_rtasks = pinned_alloc<ReconTask>(cap);
		b->d_rtasks = dev_alloc<ReconTask>(cap);
		b->rtask_cap = cap;
	}
}

void ensure_chunk_events(Batch *b, size_t n) {
	while (b->ev_info.size() < n) {
		cudaEvent_t e = nullptr;
		CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
		b->ev_info.push_back(e);
	}
	while (b->ev_rec0.size() < n) {
		cudaEvent_t e = nullptr;
		CUDA_CHECK(cudaEventCreate(&e));
		b->ev_rec0.push_back(e);
	}
	while (b->ev_rec1.size() < n) {
		cudaEvent_t e = nullptr;
		CUDA_CHECK(cudaEventCreate(&e));
		b->ev_rec1.push_back(e);
	}
}

PlaneSet plane_set(const Stream &s, uint8_t *base) {
	PlaneSet p;
	p.y = base;
	p.cr = base + s.coded_size;
	p.cb = base + s.coded_size + (s.coded_size >> 2);
	return p;
}

bool entry_stale(const Stream &s, const Parsed &e) {
	// a parse that ran into the end of the data it saw must be redone once more data is there (SURVEY Q15)
	return e.len_at_parse != s.bb.length && (uint64_t)e.info.end_bit + 64 >= (uint64_t)e.len_at_parse * 8;
}

// The copy-out of one reconstruct launch's pictures (OUT_HOST), on the copy stream.
void copy_out_step(Batch *b, const std::vector<ReconTask> &tasks, const std::vector<int> &stream_ids) {
	CUDA_CHECK(cudaEventRecord(b->ev_step, b->st_recon));
	CUDA_CHECK(cudaStreamWaitEvent(b->st_copy, b->ev_step, 0));
	// all pictures of the step leave in ONE batched copy call (cudaMemcpyBatchAsync, CUDA 12.8+)
	const size_t n_copy = tasks.size();
	b->copy_dst.resize(n_copy);
	b->copy_src.resize(n_copy);
	b->copy_size.resize(n_copy);
	for (size_t i = 0; i < n_copy; i++) {
		Stream &s = b->streams[stream_ids[i]];
		s.h_head = (s.h_head + 1) % HOST_RING;
		b->copy_dst[i] = s.h_planes[s.h_head];
		b->copy_src[i] = tasks[i].cur.y;
		b->copy_size[i] = (size_t)s.coded_size * 3 / 2;
		b->stats.d2h_bytes += b->copy_size[i];
	}
	bool batched = false;
	if (b->batch_copy_ok && n_copy > 1) {
		cudaMemcpyAttributes attr{};
		attr.srcAccessOrder = cudaMemcpySrcAccessOrderStream;
		size_t attr_idx = 0, fail_idx = 0;
		cudaError_t e = cudaMemcpyBatchAsync(b->copy_dst.data(), b->copy_src.data(), b->copy_size.data(), n_copy,
		                                     &attr, &attr_idx, 1, &fail_idx, b->st_copy);
		if (e == cudaSuccess) batched = true;
		else { (void)cudaGetLastError(); b->batch_copy_ok = false; }  // older driver: plain copies from now on
	}
	if (!batched)
		for (size_t i = 0; i < n_copy; i++)
			CUDA_CHECK(cudaMemcpyAsync(b->copy_dst[i], b->copy_src[i], b->copy_size[i], cudaMemcpyDeviceToHost, b->st_copy));
	CUDA_CHECK(cudaEventRecord(b->ev_copied[b->copy_steps & 1], b->st_copy));
	b->copy_steps++;
}

// One round: parse ahead what is missing (one wave, queued chunk by chunk), then -- chunk after chunk, as
// the chunks' infos arrive -- consume up to want[s] pictures per stream in decode() order and queue their
// reconstruction.  Returns pictures consumed; `progress[s]` gets the per-stream count, `more[s]` whether
// the stream may have further pictures.
long decode_round(Batch *b, const std::vector<int> &want, std::vector<int> &progress, std::vector<char> &more, int flags) {
	const int S = (int)b->streams.size();
	// ---- 1. plan the parse wave
	// kind: which walk kernel takes the picture -- 0 the lane-parallel walk, 1 the slice walk, 2 the B-picture walk
	struct NewParse { int stream; size_t cache_idx; uint32_t bytes; int chunk; uint32_t pic; int kind; };
	std::vector<NewParse> fresh;
	for (int si = 0; si < S; si++) {
		Stream &s = b->streams[si];
		progress[si] = 0;
		if (!s.has_seq || want[si] <= 0) { more[si] = 0; continue; }
		const uint32_t from_byte = (s.bb.index + 7) >> 3;
		auto it = std::lower_bound(s.pics.begin(), s.pics.end(), from_byte);
		if (!s.cache.empty() && (it == s.pics.end() || s.cache.front().pos != *it)) flush_cache(b, s);
		for (size_t j = 0; j < s.cache.size(); j++) {
			if (entry_stale(s, s.cache[j])) {
				while (s.cache.size() > j) { release_slot(b, s.cache.back().slot); s.cache.pop_back(); }
				break;
			}
		}
		if ((int)s.cache.size() >= want[si]) continue;
		int target = std::max(want[si], b->lookahead);
		auto next = it + (ptrdiff_t)s.cache.size();
		// `it` may be end(); cache is then empty
		while ((int)s.cache.size() < target && next < s.pics.end() && !b->free_slots.empty()) {
			Parsed p{};
			p.pos = *next;
			p.len_at_parse = s.bb.length;
			p.slot = b->free_slots.back();
			p.ready = false;
			b->free_slots.pop_back();
			s.cache.push_back(p);
			++next;
			// the extension: a picture whose header says type 3 (ISO 11172-2 2.4.2.5: 10 bits temporal_reference, 3 bits
			// picture_coding_type) goes to the B-picture walk; everything else, and everything without it, to the I/P walk
			const int type = (uint64_t)p.pos + 5 < s.bb.length ? (s.bb.bytes[p.pos + 5] >> 3) & 7 : 0;
			const uint32_t pic = (uint32_t)(next - 1 - s.pics.begin());
			int kind = (b->decode_b && type == 3) ? 2 : 0;
			if (b->slice_walk && (type == 1 || type == 2)) {  // enough slice start codes between this picture's and the next one's?
				const uint32_t hi = pic + 1 < s.pic_code.size() ? s.pic_code[pic + 1] : (uint32_t)s.codes.size();
				int n_slices = 0;
				for (uint32_t k = s.pic_code[pic] + 1; k < hi && n_slices < SLICE_WALK_MIN_SLICES; k++) {
					const uint32_t q = s.codes[k];
					if (q + 3u < s.bb.length && s.bb.bytes[q + 3u] >= 0x01 && s.bb.bytes[q + 3u] <= 0xAF) n_slices++;
				}
				if (n_slices >= SLICE_WALK_MIN_SLICES) kind = 1;
			}
			fresh.push_back({si, s.cache.size() - 1, (next < s.pics.end() ? *next : s.bb.length) - p.pos, 0, pic, kind});
		}
	}
	// ---- 2. chunks by picture ordinal (position in the stream's look-ahead); a small wave stays whole
	const int G = (b->chunk_pictures > 0 && (int)fresh.size() >= b->chunk_min_wave) ? b->chunk_pictures : 0;
	int n_chunks = 1;
	if (G > 0) {
		for (auto &f : fresh) { f.chunk = (int)(f.cache_idx / (size_t)G); n_chunks = std::max(n_chunks, f.chunk + 1); }
		int max_ordinal = 0;
		for (int si = 0; si < S; si++) max_ordinal = std::max(max_ordinal, std::max(want[si], 0));
		n_chunks = std::max(n_chunks, (max_ordinal + G - 1) / G);
	}
	ensure_chunk_events(b, (size_t)n_chunks);
	std::vector<int> chunk_off(n_chunks + 1, 0);
	if (!fresh.empty()) {
		// Within a chunk, longest pictures first: a CTA's warps, and consecutive CTAs (which land on different
		// SMs), then carry similar amounts of work and the chunk's walk ends without a long tail.
		// (and grouped by the walk kernel that takes them)
		std::stable_sort(fresh.begin(), fresh.end(), [](const NewParse &x, const NewParse &y) {
			return x.chunk != y.chunk ? x.chunk < y.chunk : (x.kind != y.kind ? x.kind < y.kind : x.bytes > y.bytes);
		});
		for (auto &f : fresh) chunk_off[f.chunk + 1]++;
		for (int c = 0; c < n_chunks; c++) chunk_off[c + 1] += chunk_off[c];
		ensure_task_caps(b, (int)fresh.size(), 0);
		for (size_t i = 0; i < fresh.size(); i++) {
			Stream &s = b->streams[fresh[i].stream];
			Parsed &p = s.cache[fresh[i].cache_idx];
			ParseTask &t = b->h_ptasks[i];
			t.es = s.d_es;
			t.es_len = s.bb.length;
			t.start_byte = p.pos + 4;
			t.seq = s.d_seq;
			t.hdr = b->d_hdr + (size_t)p.slot * b->slot_mb;
			t.coef = b->d_coef + (size_t)p.slot * b->slot_mb * MB_COEF_INT16;
			t.park = b->d_park + (size_t)p.slot * b->slot_mb * 6;
			t.info = b->d_info + i;
			t.mb_width = s.seq.mb_width;
			t.mb_size = s.seq.mb_size;
			t.stage = b->d_stage + (size_t)p.slot * stage_entries_for(b->slot_mb) * 4;
			t.stage_entries = stage_entries_for(b->slot_mb);
			t.codes = b->d_codes ? b->d_codes + (size_t)fresh[i].stream * b->codes_stride : nullptr;
			t.n_codes = (uint32_t)s.codes.size();
			t.code_hint = s.pic_code[fresh[i].pic];
		}
		if (b->recon_pending) {  // slots freed by the previous round are still being read by its reconstruct launches
			CUDA_CHECK(cudaStreamWaitEvent(b->st_main, b->ev_round, 0));
			b->recon_pending = false;
		}
		CUDA_CHECK(cudaMemcpyAsync(b->d_ptasks, b->h_ptasks, fresh.size() * sizeof(ParseTask), cudaMemcpyHostToDevice, b->st_main));
		CUDA_CHECK(cudaEventRecord(b->ev_a, b->st_main));
		// Chunks are parsed on a few streams in turn: the walk of chunk c + 1 starts while chunk c is still walking or
		// expanding (a chunk's walk costs its latency floor whatever its size; in a row on one stream the floors add up).
		const int n_cs = (G > 0 && n_chunks > 1) ? std::min(std::max(b->chunk_streams, 1), 4) : 1;
		if (n_cs > 1) {
			for (int k = 0; k < n_cs; k++)
				if (!b->st_chunk[k]) {
					CUDA_CHECK(cudaStreamCreateWithFlags(&b->st_chunk[k], cudaStreamNonBlocking));
					CUDA_CHECK(cudaEventCreateWithFlags(&b->ev_chunk_done[k], cudaEventDisableTiming));
				}
			if (!b->ev_fed) CUDA_CHECK(cudaEventCreateWithFlags(&b->ev_fed, cudaEventDisableTiming));
			CUDA_CHECK(cudaEventRecord(b->ev_fed, b->st_main));  // tasks uploaded, the previous round's reconstruction waited for
		}
		bool mid_recorded = false;
		for (int c = 0; c < n_chunks; c++) {
			const int lo = chunk_off[c], n = chunk_off[c + 1] - lo;
			cudaStream_t st = n_cs > 1 ? b->st_chunk[c % n_cs] : b->st_main;
			if (n_cs > 1 && c < n_cs) CUDA_CHECK(cudaStreamWaitEvent(st, b->ev_fed, 0));
			if (n > 0) {
				// the chunk's pictures by walk kernel: [lo, lo + cnt[0]) lane-parallel walk, then the slice walk's, then the B pictures
				int cnt[3] = {0, 0, 0};
				for (int i = lo; i < lo + n; i++) cnt[fresh[i].kind]++;
				const int off[3] = {lo, lo + cnt[0], lo + cnt[0] + cnt[1]};
				// The first kind present stays on `st`; the others have walk kernels of their own (one warp per picture,
				// latency-bound like every walk) and run beside it on side streams, forked before anything is queued and
				// joined before the infos are read.
				int primary = 0;
				while (cnt[primary] == 0) primary++;
				const bool side = cnt[0] + cnt[1] + cnt[2] > cnt[primary];
				if (side) {
					if (!b->ev_sfork) {
						CUDA_CHECK(cudaEventCreateWithFlags(&b->ev_sfork, cudaEventDisableTiming));
						for (int j = 0; j < 2; j++) {
							CUDA_CHECK(cudaStreamCreateWithFlags(&b->st_side[j], cudaStreamNonBlocking));
							CUDA_CHECK(cudaEventCreateWithFlags(&b->ev_sjoin[j], cudaEventDisableTiming));
						}
					}
					CUDA_CHECK(cudaEventRecord(b->ev_sfork, st));
				}
				int n_side = 0;
				for (int kind = 0; kind < 3; kind++) {
					if (cnt[kind] == 0) continue;
					cudaStream_t sk = st;
					if (kind != primary) {
						sk = b->st_side[n_side];
						CUDA_CHECK(cudaStreamWaitEvent(sk, b->ev_sfork, 0));
					}
					if (kind == 0) {
						launch_parse_pictures(b->d_ptasks + off[0], cnt[0], b->slot_mb, sk, mid_recorded ? nullptr : b->ev_mid, n_cs > 1 ? nullptr : &b->fork);
						mid_recorded = true;
						b->stats.kernel_launches += 2 * parse_group_count(cnt[0], n_cs == 1);  // walk + expand per size group
					} else {
						if (kind == 1) launch_parse_pictures_slices(b->d_ptasks + off[1], cnt[1], b->slot_mb, sk);
						else launch_parse_pictures_b(b->d_ptasks + off[2], cnt[2], b->slot_mb, sk);
						b->stats.kernel_launches += 2;
					}
					if (kind != primary) {
						CUDA_CHECK(cudaEventRecord(b->ev_sjoin[n_side], sk));
						CUDA_CHECK(cudaStreamWaitEvent(st, b->ev_sjoin[n_side], 0));
						n_side++;
					}
				}
				CUDA_CHECK(cudaMemcpyAsync(b->h_info + lo, b->d_info + lo, n * sizeof(picture_info_t), cudaMemcpyDeviceToHost, st));
			}
			CUDA_CHECK(cudaEventRecord(b->ev_info[c], st));
		}
		if (n_cs > 1)  // everything queued later on the main stream comes after the whole wave
			for (int k = 0; k < n_cs; k++) {
				CUDA_CHECK(cudaEventRecord(b->ev_chunk_done[k], b->st_chunk[k]));
				CUDA_CHECK(cudaStreamWaitEvent(b->st_main, b->ev_chunk_done[k], 0));
			}
		if (!mid_recorded) CUDA_CHECK(cudaEventRecord(b->ev_mid, b->st_main));  // (a wave of B pictures only)
		CUDA_CHECK(cudaEventRecord(b->ev_b, b->st_main));
		b->stats.h2d_bytes += fresh.size() * sizeof(ParseTask);
		b->stats.d2h_bytes += fresh.size() * sizeof(picture_info_t);
	}
	// ---- 3. chunk after chunk: absorb the infos, consume in decode() order, queue the reconstruction
	long consumed = 0;
	std::vector<char> open(S, 0);  // stream still consuming in this round
	std::vector<int> taken(S, 0);  // pictures consumed (= ordinal of the stream's next picture)
	for (int si = 0; si < S; si++) {
		const Stream &s = b->streams[si];
		if (s.has_seq && want[si] > 0) { open[si] = 1; more[si] = 1; }
	}
	int rec_chunks = 0;
	for (int c = 0; c < n_chunks; c++) {
		const int lo = chunk_off[c], n = chunk_off[c + 1] - lo;
		if (n > 0) {
			CUDA_CHECK(cudaEventSynchronize(b->ev_info[c]));
			for (int i = lo; i < lo + n; i++) {
				Stream &s = b->streams[fresh[i].stream];
				// cache indices were taken at planning time; `taken` pictures have left the front since
				const size_t tk = (size_t)taken[fresh[i].stream];
				if (fresh[i].cache_idx < tk || fresh[i].cache_idx - tk >= s.cache.size()) continue;  // flushed meanwhile
				Parsed &p = s.cache[fresh[i].cache_idx - tk];
				p.info = b->h_info[i];
				p.ready = true;
				if (p.info.error == PARSE_ERR_INVALID_VLC) b->stats.parse_errors++;
				if (p.info.reserved[0]) b->stats.lane_walk_pictures++;
			}
		}
		// step j of a stream -> reconstruct launch j of the chunk
		std::vector<std::vector<ReconTask>> steps;
		std::vector<std::vector<int>> step_streams;
		const int ordinal_end = G > 0 ? (c + 1) * G : 0x7fffffff;
		for (int si = 0; si < S; si++) {
			if (!open[si]) continue;
			Stream &s = b->streams[si];
			int step = 0;
			while (taken[si] < want[si] && taken[si] < ordinal_end) {
				const uint32_t from_byte = (s.bb.index + 7) >> 3;
				auto it = std::lower_bound(s.pics.begin(), s.pics.end(), from_byte);
				if (it == s.pics.end()) {  // findStartCode(PICTURE) == -1: index parks at the end (buffer.js:126-127)
					s.bb.index = s.bb.length << 3;
					more[si] = 0;
					open[si] = 0;
					break;
				}
				if (s.cache.empty() || !s.cache.front().ready || s.cache.front().pos != *it || entry_stale(s, s.cache.front())) {
					// the look-ahead does not match the serial order: re-plan in the next round.  (Entries of later
					// chunks may still be in flight; their slots are reused only by parses queued behind them.)
					flush_cache(b, s);
					open[si] = 0;
					taken[si] = 0x40000000;  // nothing of this stream's planning-time indices is valid any more
					break;
				}
				const Parsed e = s.cache.front();
				s.cache.pop_front();
				s.bb.index = e.info.end_bit;
				taken[si]++;
				progress[si]++;
				consumed++;
				b->stats.pictures++;
				b->stats.es_bytes += (e.info.end_bit >> 3) - e.pos;
				s.last_type = e.info.picture_type;
				s.last_temporal = (uint64_t)e.pos + 5 < s.bb.length ? (s.bb.bytes[e.pos + 4] << 2 | s.bb.bytes[e.pos + 5] >> 6) : 0;
				if (e.info.status == PIC_DECODED) {
					const bool is_b = e.info.picture_type == 3;  // (only the extension's walk answers PIC_DECODED for one)
					ReconTask t{};
					t.hdr = b->d_hdr + (size_t)e.slot * b->slot_mb;
					t.coef = b->d_coef + (size_t)e.slot * b->slot_mb * MB_COEF_INT16;
					if (is_b) {
						// after the swaps `cur` holds the older and `1 - cur` the newer of the two most recent I/P pictures:
						// the B picture's forward (past) and backward (future) reference.  It goes to a set of its own.
						if (!s.d_planes_b[0]) {
							const size_t bytes = (size_t)s.coded_size * 3 / 2 + s.seq.coded_width + 64;
							for (auto &pb : s.d_planes_b) {
								pb = dev_alloc<uint8_t>(bytes);
								CUDA_CHECK(cudaMemsetAsync(pb, 0, bytes, b->st_recon));
							}
						}
						t.cur = plane_set(s, s.d_planes_b[s.b_cur]);
						t.fwd = plane_set(s, s.d_planes[s.cur]);
						t.bwd = plane_set(s, s.d_planes[1 - s.cur]);
					} else {
						t.cur = plane_set(s, s.d_planes[s.cur]);
						t.fwd = plane_set(s, s.d_planes[1 - s.cur]);
					}
					s.d_last = t.cur.y;
					t.mb_width = s.seq.mb_width;
					t.mb_size = s.seq.mb_size;
					t.coded_width = s.seq.coded_width;
					t.coded_height = s.seq.coded_height;
					t.width = s.width;
					t.height = s.height;
					t.rgba = nullptr;
					if (flags & JSMPEG_B200_OUT_RGBA) {
						if (!s.d_rgba) {  // opaque white, like the canvas the reference creates (canvas2d.js:24-29): the odd edge keeps it
							s.d_rgba = dev_alloc<uint8_t>((size_t)s.width * s.height * 4);
							CUDA_CHECK(cudaMemsetAsync(s.d_rgba, 0xff, (size_t)s.width * s.height * 4, b->st_recon));
						}
						t.rgba = s.d_rgba;
					}
					if ((int)steps.size() <= step) { steps.emplace_back(); step_streams.emplace_back(); }
					steps[step].push_back(t);
					step_streams[step].push_back(si);
					step++;
					if (is_b) s.b_cur ^= 1;  // no reference: the I/P ping-pong stays as it is
					else s.cur ^= 1;         // mpeg1.js:221-246: the picture just decoded becomes `forward`
					b->stats.pictures_decoded++;
					b->stats.coded_blocks += e.info.n_coded_blocks;
					b->stats.macroblocks += e.info.n_present;
					const uint64_t planes = (uint64_t)s.coded_size * 3 / 2;
					b->stats.algorithmic_bytes += planes + (e.info.picture_type == 2 ? planes : (is_b ? 2 * planes : 0)) +
					                              (uint64_t)s.seq.mb_size * sizeof(mb_record_t) + (uint64_t)e.info.n_coded_blocks * 128;
				}
				release_slot(b, e.slot);  // reused by the NEXT round's parse, which waits for this round's reconstruction (ev_round)
			}
			if (open[si] && taken[si] >= want[si]) open[si] = 0;
		}
		// ---- 4. reconstruction of the chunk, one launch per step, on the reconstruct stream
		if (steps.empty()) continue;
		size_t total = 0;
		for (auto &v : steps) total += v.size();
		ensure_task_caps(b, 0, (int)total);
		size_t off = 0;
		std::vector<int> step_n_b(steps.size(), 0);
		for (size_t f = 0; f < steps.size(); f++) {
			auto &v = steps[f];
			// the step's B pictures (extension) behind its I/P pictures: they take the two-reference kernel
			int n_b = 0;
			for (auto &t : v) n_b += t.bwd.y != nullptr;
			if (n_b) {
				std::vector<ReconTask> tv;
				std::vector<int> sv;
				for (int pass = 0; pass < 2; pass++)
					for (size_t i = 0; i < v.size(); i++)
						if ((v[i].bwd.y != nullptr) == (pass == 1)) { tv.push_back(v[i]); sv.push_back(step_streams[f][i]); }
				v.swap(tv);
				step_streams[f].swap(sv);
			}
			step_n_b[f] = n_b;
			memcpy(b->h_rtasks + off, v.data(), v.size() * sizeof(ReconTask));
			off += v.size();
		}
		CUDA_CHECK(cudaEventRecord(b->ev_rec0[rec_chunks], b->st_recon));
		off = 0;
		for (size_t f = 0; f < steps.size(); f++) {
			// A launch overwrites, per stream, the plane set written two of that stream's pictures ago, i.e. by
			// a launch at least two copy-out launches back: the copy-out recorded two launches ago must be done
			// (the copy stream is in order, so that covers every earlier one).
			if ((flags & JSMPEG_B200_OUT_HOST) && b->copy_steps >= 2)
				CUDA_CHECK(cudaStreamWaitEvent(b->st_recon, b->ev_copied[b->copy_steps & 1], 0));
			const int n_ip = (int)steps[f].size() - step_n_b[f];
			if (n_ip > 0) {
				if (flags & JSMPEG_B200_OUT_RGBA) launch_reconstruct_rgba(b->h_rtasks + off, n_ip, b->st_recon);  // conversion fused in
				else launch_reconstruct(b->h_rtasks + off, n_ip, b->st_recon);
				b->stats.kernel_launches += (n_ip + (flags & JSMPEG_B200_OUT_RGBA ? 59 : 79)) / (flags & JSMPEG_B200_OUT_RGBA ? 60 : 80);
			}
			if (step_n_b[f] > 0)
				b->stats.kernel_launches += launch_reconstruct_b(b->h_rtasks + off + n_ip, step_n_b[f], (flags & JSMPEG_B200_OUT_RGBA) != 0, b->st_recon);
			b->stats.recon_launches++;
			if (flags & JSMPEG_B200_OUT_HOST) copy_out_step(b, steps[f], step_streams[f]);  // while the next step reconstructs
			off += steps[f].size();
		}
		CUDA_CHECK(cudaEventRecord(b->ev_rec1[rec_chunks], b->st_recon));
		rec_chunks++;
		// h_rtasks is read at launch time only (the table travels in the kernel parameters), so the next chunk may reuse it
	}
	if (rec_chunks) {
		CUDA_CHECK(cudaEventRecord(b->ev_round, b->st_recon));
		b->recon_pending = true;
		CUDA_CHECK(cudaEventSynchronize(b->ev_rec1[rec_chunks - 1]));
		for (int k = 0; k < rec_chunks; k++) {
			float ms = 0;
			CUDA_CHECK(cudaEventElapsedTime(&ms, b->ev_rec0[k], b->ev_rec1[k]));
			b->stats.recon_ms += ms;
		}
	}
	if (!fresh.empty()) {
		CUDA_CHECK(cudaEventSynchronize(b->ev_b));
		float ms = 0;
		CUDA_CHECK(cudaEventElapsedTime(&ms, b->ev_a, b->ev_b));
		b->stats.parse_ms += ms;
		CUDA_CHECK(cudaEventElapsedTime(&ms, b->ev_a, b->ev_mid));
		b->stats.walk_ms += ms;
	}
	return consumed;
}

long batch_decode(Batch *b, int n_pictures, int flags) {
	use_device(b);
	upload_all(b);
	ensure_pool(b);
	const int S = (int)b->streams.size();
	std::vector<int> remaining(S, n_pictures), want(S), progress(S);
	std::vector<char> more(S, 1);
	long total = 0;
	int idle_rounds = 0;
	for (;;) {
		int active = 0;
		for (int i = 0; i < S; i++) if (more[i] && remaining[i] > 0 && b->streams[i].has_seq) active++;
		if (!active) break;
		// share the record slots between the active streams
		int cached = 0;
		for (auto &s : b->streams) cached += (int)s.cache.size();
		const int per_stream = std::max(1, (int)(b->free_slots.size() + cached) / active);
		for (int i = 0; i < S; i++)
			want[i] = (more[i] && b->streams[i].has_seq) ? std::min(remaining[i], per_stream) : 0;
		const long got = decode_round(b, want, progress, more, flags);
		total += got;
		bool replanned = false;
		for (int i = 0; i < S; i++) {
			remaining[i] -= progress[i];
			if (want[i] > 0 && progress[i] < want[i] && more[i]) replanned = true;
		}
		if (got == 0 && (!replanned || ++idle_rounds > 2)) break;
		if (got) idle_rounds = 0;
	}
	CUDA_CHECK(cudaStreamSynchronize(b->st_recon));
	CUDA_CHECK(cudaStreamSynchronize(b->st_copy));
	CUDA_CHECK(cudaStreamSynchronize(b->st_main));
	b->recon_pending = false;
	return total;
}

int env_int(const char *name, int fallback) {
	const char *e = getenv(name);
	return e && *e ? atoi(e) : fallback;
}

}  // namespace

// ================================================================================================
// C ABI, part 2 (batch)

extern "C" {

const char *jsmpeg_b200_version(void) { return "jsmpeg_b200 0.2 (sm_100a)"; }

jsmpeg_b200_batch_t *jsmpeg_b200_batch_create(int n_streams, int device, unsigned int max_slots) {
	Batch *b = new Batch();
	b->device = device;
	b->streams.resize(std::max(n_streams, 1));
	b->max_slots_req = max_slots;
	b->chunk_pictures = std::max(0, env_int("JSMPEG_B200_CHUNK", 0));
	b->chunk_min_wave = std::max(1, env_int("JSMPEG_B200_CHUNK_MIN_WAVE", 256));
	b->chunk_streams = std::min(std::max(1, env_int("JSMPEG_B200_CHUNK_STREAMS", 3)), 4);
	b->decode_b = env_int("JSMPEG_B200_DECODE_B", 0) != 0;
	b->slice_walk = env_int("JSMPEG_B200_SLICE_WALK", 0) != 0;
	try {
		use_device(b);
		CUDA_CHECK(cudaStreamCreateWithFlags(&b->st_main, cudaStreamNonBlocking));
		CUDA_CHECK(cudaStreamCreateWithFlags(&b->st_recon, cudaStreamNonBlocking));
		CUDA_CHECK(cudaStreamCreateWithFlags(&b->st_copy, cudaStreamNonBlocking));
		cudaEvent_t *evs[] = {&b->ev_a, &b->ev_b, &b->ev_mid};
		for (auto e : evs) CUDA_CHECK(cudaEventCreate(e));
		CUDA_CHECK(cudaEventCreateWithFlags(&b->ev_step, cudaEventDisableTiming));
		CUDA_CHECK(cudaEventCreateWithFlags(&b->ev_round, cudaEventDisableTiming));
		for (auto &e : b->ev_copied) CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
		CUDA_CHECK(cudaEventCreateWithFlags(&b->fork.fork, cudaEventDisableTiming));
		for (int i = 0; i < PARSE_GROUPS; i++) {
			CUDA_CHECK(cudaStreamCreateWithFlags(&b->fork.side[i], cudaStreamNonBlocking));
			CUDA_CHECK(cudaEventCreateWithFlags(&b->fork.join[i], cudaEventDisableTiming));
		}
	} catch (const std::exception &e) {
		mark_dead(b, e.what());  // no usable device: a decoder that answers false, not a dead process
	}
	return b;
}

void jsmpeg_b200_batch_destroy(jsmpeg_b200_batch_t *b) {
	if (!b) return;
	// best effort, nothing here may throw: the context may be the very thing that failed
	(void)cudaSetDevice(b->device);
	(void)cudaDeviceSynchronize();
	for (auto &s : b->streams) {
		if (s.bb.bytes) cudaFreeHost(s.bb.bytes);
		if (s.d_seq) cudaFree(s.d_seq);
		if (s.d_es) cudaFree(s.d_es);
		if (s.d_rgba) cudaFree(s.d_rgba);
		for (auto p : s.d_planes) if (p) cudaFree(p);
		for (auto p : s.d_planes_b) if (p) cudaFree(p);
		for (auto p : s.h_planes) if (p) cudaFreeHost(p);
	}
	if (b->d_spans) cudaFree(b->d_spans);
	if (b->h_spans) cudaFreeHost(b->h_spans);
	if (b->d_scan_counts) cudaFree(b->d_scan_counts);
	if (b->h_scan_counts) cudaFreeHost(b->h_scan_counts);
	if (b->d_scan_pos) cudaFree(b->d_scan_pos);
	if (b->h_scan_pos) cudaFreeHost(b->h_scan_pos);
	if (b->d_codes) cudaFree(b->d_codes);
	if (b->h_codes) cudaFreeHost(b->h_codes);
	if (b->d_hdr) cudaFree(b->d_hdr);
	if (b->d_coef) cudaFree(b->d_coef);
	if (b->d_park) cudaFree(b->d_park);
	if (b->d_stage) cudaFree(b->d_stage);
	if (b->d_info) cudaFree(b->d_info);
	if (b->h_info) cudaFreeHost(b->h_info);
	if (b->h_ptasks) cudaFreeHost(b->h_ptasks);
	if (b->d_ptasks) cudaFree(b->d_ptasks);
	if (b->h_rtasks) cudaFreeHost(b->h_rtasks);
	if (b->d_rtasks) cudaFree(b->d_rtasks);
	ts_scratch_destroy(b->ts);
	cudaEvent_t evs[] = {b->ev_a, b->ev_b, b->ev_mid, b->ev_step, b->ev_round, b->ev_copied[0], b->ev_copied[1], b->fork.fork};
	for (auto e : evs) if (e) cudaEventDestroy(e);
	for (auto v : {&b->ev_info, &b->ev_rec0, &b->ev_rec1}) for (auto e : *v) if (e) cudaEventDestroy(e);
	for (int i = 0; i < PARSE_GROUPS; i++) {
		if (b->fork.join[i]) cudaEventDestroy(b->fork.join[i]);
		if (b->fork.side[i]) cudaStreamDestroy(b->fork.side[i]);
	}
	for (auto st : {b->st_main, b->st_recon, b->st_copy, b->st_side[0], b->st_side[1], b->st_chunk[0], b->st_chunk[1], b->st_chunk[2], b->st_chunk[3]}) if (st) cudaStreamDestroy(st);
	for (auto e : {b->ev_fed, b->ev_sfork, b->ev_sjoin[0], b->ev_sjoin[1], b->ev_chunk_done[0], b->ev_chunk_done[1], b->ev_chunk_done[2], b->ev_chunk_done[3]}) if (e) cudaEventDestroy(e);
	(void)cudaGetLastError();
	delete b;
}

const char *jsmpeg_b200_batch_last_error(jsmpeg_b200_batch_t *b) { return (b && b->dead) ? b->error.c_str() : nullptr; }

int jsmpeg_b200_batch_set_option(jsmpeg_b200_batch_t *b, const char *name, int value) {
	if (!b || !name) return -1;
	if (!strcmp(name, "chunk_pictures")) { b->chunk_pictures = std::max(0, value); return 0; }
	if (!strcmp(name, "chunk_min_wave")) { b->chunk_min_wave = std::max(1, value); return 0; }
	if (!strcmp(name, "chunk_streams")) { b->chunk_streams = std::min(std::max(1, value), 4); return 0; }
	if (!strcmp(name, "lookahead")) { b->lookahead = std::max(1, value); return 0; }
	if (!strcmp(name, "slice_walk")) { b->slice_walk = value != 0; return 0; }  // (same records either way: nothing to flush)
	if (!strcmp(name, "decode_b")) {
		if (b->decode_b != (value != 0))
			for (auto &st : b->streams) flush_cache(b, st);  // what was parsed ahead was parsed under the other rule
		b->decode_b = value != 0;
		return 0;
	}
	return -1;
}

void *jsmpeg_b200_batch_get_write_ptr(jsmpeg_b200_batch_t *b, int stream, unsigned int byte_size) {
	void *p = guarded<void *>(b, nullptr, [&]() -> void * {
		use_device(b);
		return stream_get_write_ptr(b, b->streams[stream], byte_size);
	});
	if (p) return p;
	// dead decoder: the caller's memcpy still needs somewhere to go
	b->dead_scratch.resize(std::max<size_t>(byte_size, 1));
	return b->dead_scratch.data();
}

void jsmpeg_b200_batch_did_write(jsmpeg_b200_batch_t *b, int stream, unsigned int byte_size) {
	guarded_void(b, [&] {
		use_device(b);
		stream_did_write(b, b->streams[stream], byte_size);
	});
}

int jsmpeg_b200_batch_get_index(jsmpeg_b200_batch_t *b, int stream) { return (int)b->streams[stream].bb.index; }

void jsmpeg_b200_batch_set_index(jsmpeg_b200_batch_t *b, int stream, unsigned int index) {
	Stream &s = b->streams[stream];
	s.bb.index = index;
	flush_cache(b, s);
}

int jsmpeg_b200_batch_stream_info(jsmpeg_b200_batch_t *b, int stream, int *width, int *height, int *coded_size, float *frame_rate) {
	const Stream &s = b->streams[stream];
	if (width) *width = s.width;
	if (height) *height = s.height;
	if (coded_size) *coded_size = s.coded_size;
	if (frame_rate) *frame_rate = s.frame_rate;
	return s.has_seq ? 1 : 0;
}

long jsmpeg_b200_batch_upload(jsmpeg_b200_batch_t *b) {
	return guarded<long>(b, 0, [&] {
		use_device(b);
		return upload_all(b);
	});
}

void jsmpeg_b200_batch_rewind(jsmpeg_b200_batch_t *b) {
	for (auto &s : b->streams) {
		flush_cache(b, s);
		s.pics.clear();
		s.codes.clear();
		s.pic_code.clear();
		s.codes_classified = 0;
		s.scanned = 0;
		s.bb.index = s.has_seq ? s.seq_end_index : 0;  // where did_write left it (mpeg1.c:812-819)
	}
}

void jsmpeg_b200_batch_reset(jsmpeg_b200_batch_t *b) {
	guarded_void(b, [&] {
		use_device(b);
		for (auto &s : b->streams) {
			forget_index(b, s);
			s.bb.length = 0;
			s.bb.index = 0;
			s.cur = 0;
			s.b_cur = 0;
			s.d_last = nullptr;
			s.last_type = s.last_temporal = 0;
			s.h_head = -1;
			if (s.has_seq) {
				for (auto p : s.d_planes) CUDA_CHECK(cudaMemsetAsync(p, 0, (size_t)s.coded_size * 3 / 2, b->st_main));
				for (auto p : s.d_planes_b) if (p) CUDA_CHECK(cudaMemsetAsync(p, 0, (size_t)s.coded_size * 3 / 2, b->st_main));
			}
		}
		CUDA_CHECK(cudaStreamSynchronize(b->st_main));
	});
}

long jsmpeg_b200_batch_decode(jsmpeg_b200_batch_t *b, int n_pictures, int flags) {
	return guarded<long>(b, 0, [&] { return batch_decode(b, n_pictures, flags); });
}

int jsmpeg_b200_batch_get_planes(jsmpeg_b200_batch_t *b, int stream, void **y, void **cr, void **cb) {
	const Stream &s = b->streams[stream];
	if (!s.has_seq) return -1;
	// most recent picture = forward (mpeg1.c:841-851); with the B-picture extension it may be a B picture's own set
	PlaneSet p = plane_set(s, s.d_last ? s.d_last : s.d_planes[1 - s.cur]);
	if (y) *y = p.y;
	if (cr) *cr = p.cr;
	if (cb) *cb = p.cb;
	return 0;
}

int jsmpeg_b200_batch_get_host_planes(jsmpeg_b200_batch_t *b, int stream, void **y, void **cr, void **cb) {
	const Stream &s = b->streams[stream];
	if (!s.has_seq) return -1;
	PlaneSet p = plane_set(s, s.h_planes[s.h_head < 0 ? 0 : s.h_head]);
	if (y) *y = p.y;
	if (cr) *cr = p.cr;
	if (cb) *cb = p.cb;
	return 0;
}

int jsmpeg_b200_batch_get_rgba(jsmpeg_b200_batch_t *b, int stream, void **rgba) {
	const Stream &s = b->streams[stream];
	if (!s.has_seq || !s.d_rgba) return -1;
	*rgba = s.d_rgba;
	return 0;
}

int jsmpeg_b200_batch_read_planes(jsmpeg_b200_batch_t *b, int stream, void *y, void *cr, void *cb) {
	return guarded<int>(b, -1, [&] {
		use_device(b);
		const Stream &s = b->streams[stream];
		if (!s.has_seq) return -1;
		PlaneSet p = plane_set(s, s.d_last ? s.d_last : s.d_planes[1 - s.cur]);
		if (y) CUDA_CHECK(cudaMemcpy(y, p.y, s.coded_size, cudaMemcpyDeviceToHost));
		if (cr) CUDA_CHECK(cudaMemcpy(cr, p.cr, s.coded_size >> 2, cudaMemcpyDeviceToHost));
		if (cb) CUDA_CHECK(cudaMemcpy(cb, p.cb, s.coded_size >> 2, cudaMemcpyDeviceToHost));
		return 0;
	});
}

long jsmpeg_b200_batch_write_ts(jsmpeg_b200_batch_t *b, int stream, const uint8_t *ts, size_t n_bytes, int stream_id,
                                uint64_t *pts_out, uint32_t *offset_out, int n_max, int *n_pes) {
	if (n_pes) *n_pes = 0;
	return guarded<long>(b, -1, [&]() -> long {
		use_device(b);
		Stream &s = b->streams[stream];
		if (!b->ts) b->ts = ts_scratch_create();
		if (s.ts_bound.empty()) s.ts_bound.assign(8192, 0);
		// what the previous call left over comes first (a partial packet, a resync that wanted more data: ts.js:25-41)
		const uint8_t *data = ts;
		size_t n_data = n_bytes;
		if (!s.ts_leftover.empty()) {
			s.ts_leftover.insert(s.ts_leftover.end(), ts, ts + n_bytes);
			data = s.ts_leftover.data();
			n_data = s.ts_leftover.size();
		}
		size_t consumed = 0;
		const long total = ts_demux_measure(b->ts, data, n_data, stream_id, s.ts_bound.data(), &consumed, b->st_main);
		std::vector<uint8_t> rest(data + consumed, data + n_data);  // (data may alias ts_leftover)
		if (total <= 0) { s.ts_leftover.swap(rest); return total; }
		// room in the host bit buffer (the reference's write protocol, may expand or evict) and in HBM
		uint8_t *hdst = static_cast<uint8_t *>(stream_get_write_ptr(b, s, (uint32_t)total));
		reserve_device_es(b, s, s.bb.length + (uint32_t)total);
		if (s.d_valid < s.bb.length) {  // bytes written the ordinary way that are not resident yet
			CUDA_CHECK(cudaMemcpyAsync(s.d_es + s.d_valid, s.bb.bytes + s.d_valid, s.bb.length - s.d_valid, cudaMemcpyHostToDevice, b->st_main));
			b->stats.h2d_bytes += s.bb.length - s.d_valid;
			s.d_valid = s.bb.length;
		}
		const int count = ts_demux_gather(b->ts, s.d_es, s.bb.length, pts_out, offset_out, n_max, b->st_main);
		s.ts_leftover.swap(rest);
		b->stats.kernel_launches += 7;
		b->stats.h2d_bytes += n_data;
		// the host keeps a mirror of the ES (sequence header parse, EVICT bookkeeping): copy the new bytes back
		CUDA_CHECK(cudaMemcpyAsync(hdst, s.d_es + s.bb.length, (size_t)total, cudaMemcpyDeviceToHost, b->st_main));
		CUDA_CHECK(cudaMemsetAsync(s.d_es + s.bb.length + total, 0, ES_PAD, b->st_main));
		CUDA_CHECK(cudaStreamSynchronize(b->st_main));
		b->stats.d2h_bytes += (uint64_t)total;
		stream_did_write(b, s, (uint32_t)total);
		s.d_valid = s.bb.length;
		if (n_pes) *n_pes = count;
		if (pts_out && offset_out && count > 1) {  // the device appends PES starts unordered: sort by offset
			const int m = std::min(count, n_max);
			std::vector<std::pair<uint32_t, uint64_t>> v(m);
			for (int i = 0; i < m; i++) v[i] = {offset_out[i], pts_out[i]};
			std::sort(v.begin(), v.end());
			for (int i = 0; i < m; i++) { offset_out[i] = v[i].first; pts_out[i] = v[i].second; }
		}
		return total;
	});
}

int jsmpeg_b200_batch_read_rgba(jsmpeg_b200_batch_t *b, int stream, void *rgba) {
	return guarded<int>(b, -1, [&] {
		use_device(b);
		const Stream &s = b->streams[stream];
		if (!s.has_seq || !s.d_rgba) return -1;
		CUDA_CHECK(cudaMemcpy(rgba, s.d_rgba, (size_t)s.width * s.height * 4, cudaMemcpyDeviceToHost));
		return 0;
	});
}

int jsmpeg_b200_batch_last_picture(jsmpeg_b200_batch_t *b, int stream, int *picture_type, int *temporal_reference) {
	const Stream &s = b->streams[stream];
	if (picture_type) *picture_type = s.last_type;
	if (temporal_reference) *temporal_reference = s.last_temporal;
	return s.last_type ? 0 : -1;
}

void jsmpeg_b200_batch_get_stats(jsmpeg_b200_batch_t *b, jsmpeg_b200_stats_t *out) { *out = b->stats; }
void jsmpeg_b200_batch_reset_stats(jsmpeg_b200_batch_t *b) { b->stats = jsmpeg_b200_stats_t{}; }

// ================================================================================================
// C ABI, part 1 (reference ABI): one stream, synchronous, host-visible planes

struct mpeg1_decoder_t {
	jsmpeg_b200_batch_t *b;
};

// Host placement.  The pinned bit buffers and plane rings of a decoder are touched by the host threads
// that drive it and by the GPU's copy engines; on a two-socket host a GPU hangs off ONE socket, and a
// ring on the other socket costs every D2H byte a trip over the socket interconnect (round 1: the
// 8-GPU e2e curve went flat at 4 GPUs).  This binds the CALLING THREAD -- and with it the threads it
// creates and the pages it first touches from now on -- to the CPUs of the NUMA node of `device`
// (sysfs: /sys/bus/pci/devices/<id>/numa_node, /sys/devices/system/node/node<k>/cpulist), intersected
// with the affinity it already has.  Returns the number of CPUs bound to, 0 if the node is unknown
// (nothing changed), -1 on error.  node_out (may be NULL) receives the node.
int jsmpeg_b200_bind_host_to_device(int device, int *node_out) {
	if (node_out) *node_out = -1;
	char id[32] = {0};
	if (cudaDeviceGetPCIBusId(id, sizeof id, device) != cudaSuccess) { (void)cudaGetLastError(); return -1; }
	for (char *c = id; *c; c++) if (*c >= 'A' && *c <= 'F') *c += 'a' - 'A';
	char path[128];
	snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", id);
	FILE *f = fopen(path, "r");
	int node = -1;
	if (f) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
	if (node < 0) return 0;
	snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
	f = fopen(path, "r");
	if (!f) return 0;
	cpu_set_t want, have, both;
	CPU_ZERO(&want);
	int lo, hi;
	while (fscanf(f, "%d", &lo) == 1) {  // "0-31,64-95"
		hi = lo;
		int ch = fgetc(f);
		if (ch == '-') { if (fscanf(f, "%d", &hi) != 1) hi = lo; ch = fgetc(f); }
		for (int c = lo; c <= hi && c < CPU_SETSIZE; c++) CPU_SET(c, &want);
		if (ch != ',') break;
	}
	fclose(f);
	if (sched_getaffinity(0, sizeof have, &have) != 0) return -1;
	CPU_AND(&both, &want, &have);
	const int n = CPU_COUNT(&both);
	if (n == 0) return 0;
	if (sched_setaffinity(0, sizeof both, &both) != 0) return -1;
	if (node_out) *node_out = node;
	return n;
}

static int g_default_device = -1;  // -1: JSMPEG_B200_DEVICE or 0
void jsmpeg_b200_set_default_device(int device) { g_default_device = device; }

mpeg1_decoder_t *mpeg1_decoder_create(unsigned int buffer_size, bit_buffer_mode_t buffer_mode) {
	int lookahead = env_int("JSMPEG_B200_LOOKAHEAD", 16);
	if (lookahead < 1) lookahead = 1;
	mpeg1_decoder_t *d = new mpeg1_decoder_t();
	d->b = jsmpeg_b200_batch_create(1, g_default_device >= 0 ? g_default_device : env_int("JSMPEG_B200_DEVICE", 0), (unsigned)lookahead + 1);
	d->b->lookahead = lookahead;
	Stream &s = d->b->streams[0];
	s.bb.mode = buffer_mode;
	guarded_void(d->b, [&] {
		if (!bitbuffer::resize(s.bb, buffer_size ? buffer_size : 1, kPinned)) throw std::runtime_error("jsmpeg_b200: bit buffer allocation failed");
	});
	return d;
}

void mpeg1_decoder_destroy(mpeg1_decoder_t *self) {
	if (!self) return;
	jsmpeg_b200_batch_destroy(self->b);
	delete self;
}

const char *jsmpeg_b200_decoder_last_error(mpeg1_decoder_t *self) { return self ? jsmpeg_b200_batch_last_error(self->b) : nullptr; }
int jsmpeg_b200_decoder_set_option(mpeg1_decoder_t *self, const char *name, int value) {
	return self ? jsmpeg_b200_batch_set_option(self->b, name, value) : -1;
}
int jsmpeg_b200_decoder_last_picture(mpeg1_decoder_t *self, int *picture_type, int *temporal_reference) {
	return self ? jsmpeg_b200_batch_last_picture(self->b, 0, picture_type, temporal_reference) : -1;
}

void *mpeg1_decoder_get_write_ptr(mpeg1_decoder_t *self, unsigned int byte_size) {
	return jsmpeg_b200_batch_get_write_ptr(self->b, 0, byte_size);
}
int mpeg1_decoder_get_index(mpeg1_decoder_t *self) { return jsmpeg_b200_batch_get_index(self->b, 0); }
void mpeg1_decoder_set_index(mpeg1_decoder_t *self, unsigned int index) { jsmpeg_b200_batch_set_index(self->b, 0, index); }
void mpeg1_decoder_did_write(mpeg1_decoder_t *self, unsigned int byte_size) { jsmpeg_b200_batch_did_write(self->b, 0, byte_size); }
int mpeg1_decoder_has_sequence_header(mpeg1_decoder_t *self) { return self->b->streams[0].has_seq ? 1 : 0; }
float mpeg1_decoder_get_frame_rate(mpeg1_decoder_t *self) { return self->b->streams[0].frame_rate; }
int mpeg1_decoder_get_coded_size(mpeg1_decoder_t *self) { return self->b->streams[0].coded_size; }
int mpeg1_decoder_get_width(mpeg1_decoder_t *self) { return self->b->streams[0].width; }
int mpeg1_decoder_get_height(mpeg1_decoder_t *self) { return self->b->streams[0].height; }

static void *host_plane(mpeg1_decoder_t *self, int which) {
	void *p[3] = {nullptr, nullptr, nullptr};
	if (jsmpeg_b200_batch_get_host_planes(self->b, 0, &p[0], &p[1], &p[2]) != 0) return nullptr;
	return p[which];
}
void *mpeg1_decoder_get_y_ptr(mpeg1_decoder_t *self) { return host_plane(self, 0); }
void *mpeg1_decoder_get_cr_ptr(mpeg1_decoder_t *self) { return host_plane(self, 1); }
void *mpeg1_decoder_get_cb_ptr(mpeg1_decoder_t *self) { return host_plane(self, 2); }

bool mpeg1_decoder_decode(mpeg1_decoder_t *self) {
	if (!self->b->streams[0].has_seq) return false;
	return jsmpeg_b200_batch_decode(self->b, 1, JSMPEG_B200_OUT_HOST) > 0;
}

// ================================================================================================
// test hooks

int jsmpeg_b200_debug_parse_picture(const uint8_t *es, uint32_t es_len, uint32_t start_byte, int mb_width,
                                    int mb_height, const uint8_t *intra_q, const uint8_t *non_intra_q,
                                    void *info_out, void *hdr_out, void *coef_out) {
	try {
		SeqParams sp{};
		sp.mb_width = mb_width; sp.mb_height = mb_height; sp.mb_size = mb_width * mb_height;
		sp.coded_width = mb_width * 16; sp.coded_height = mb_height * 16;
		memcpy(sp.intra_q, intra_q, 64);
		memcpy(sp.non_intra_q, non_intra_q, 64);
		seq_fill_xq(sp);
		const size_t n_mb = sp.mb_size;
		uint8_t *d_es = dev_alloc<uint8_t>(es_len + ES_PAD);
		SeqParams *d_seq = dev_alloc<SeqParams>(1);
		mb_record_t *d_hdr = dev_alloc<mb_record_t>(n_mb);
		int16_t *d_coef = dev_alloc<int16_t>(n_mb * MB_COEF_INT16);
		uint2 *d_park = dev_alloc<uint2>(n_mb * 6);
		uint4 *d_stage = dev_alloc<uint4>((size_t)stage_entries_for(sp.mb_size) * 4);
		picture_info_t *d_info = dev_alloc<picture_info_t>(1);
		ParseTask *d_task = dev_alloc<ParseTask>(1);
		CUDA_CHECK(cudaMemcpy(d_es, es, es_len, cudaMemcpyHostToDevice));
		CUDA_CHECK(cudaMemset(d_es + es_len, 0, ES_PAD));
		CUDA_CHECK(cudaMemcpy(d_seq, &sp, sizeof(sp), cudaMemcpyHostToDevice));
		CUDA_CHECK(cudaMemset(d_coef, 0, n_mb * MB_COEF_INT16 * sizeof(int16_t)));
		ParseTask t{};
		t.es = d_es; t.es_len = es_len; t.start_byte = start_byte; t.seq = d_seq; t.hdr = d_hdr; t.coef = d_coef; t.info = d_info;
		t.park = d_park; t.mb_width = mb_width; t.mb_size = sp.mb_size;
		t.stage = d_stage; t.stage_entries = stage_entries_for(sp.mb_size);
		t.codes = nullptr; t.n_codes = 0; t.code_hint = 0;  // this hook lets the walk search the slice end itself
		CUDA_CHECK(cudaMemcpy(d_task, &t, sizeof(t), cudaMemcpyHostToDevice));
		launch_parse_pictures(d_task, 1, sp.mb_size, 0);
		CUDA_CHECK(cudaGetLastError());
		CUDA_CHECK(cudaDeviceSynchronize());
		CUDA_CHECK(cudaMemcpy(info_out, d_info, sizeof(picture_info_t), cudaMemcpyDeviceToHost));
		CUDA_CHECK(cudaMemcpy(hdr_out, d_hdr, n_mb * sizeof(mb_record_t), cudaMemcpyDeviceToHost));
		CUDA_CHECK(cudaMemcpy(coef_out, d_coef, n_mb * MB_COEF_INT16 * sizeof(int16_t), cudaMemcpyDeviceToHost));
		cudaFree(d_es); cudaFree(d_seq); cudaFree(d_hdr); cudaFree(d_coef); cudaFree(d_park); cudaFree(d_stage); cudaFree(d_info); cudaFree(d_task);
		return 0;
	} catch (const std::exception &e) {
		fprintf(stderr, "%s\n", e.what());
		return -1;
	}
}

int jsmpeg_b200_debug_reconstruct(int mb_width, int mb_height, const void *hdr, const void *coef,
                                  const uint8_t *fwd_y, const uint8_t *fwd_cr, const uint8_t *fwd_cb,
                                  uint8_t *cur_y, uint8_t *cur_cr, uint8_t *cur_cb) {
	try {
		const size_t n_mb = (size_t)mb_width * mb_height;
		const size_t ysz = n_mb * 256, csz = ysz / 4, total = ysz + 2 * csz;
		mb_record_t *d_hdr = dev_alloc<mb_record_t>(n_mb);
		int16_t *d_coef = dev_alloc<int16_t>(n_mb * MB_COEF_INT16);
		const size_t pad = (size_t)mb_width * 16 + 64;
		uint8_t *d_fwd = dev_alloc<uint8_t>(total + pad), *d_cur = dev_alloc<uint8_t>(total + pad);
		CUDA_CHECK(cudaMemset(d_fwd + total, 0, pad));
		CUDA_CHECK(cudaMemcpy(d_hdr, hdr, n_mb * sizeof(mb_record_t), cudaMemcpyHostToDevice));
		CUDA_CHECK(cudaMemcpy(d_coef, coef, n_mb * MB_COEF_INT16 * sizeof(int16_t), cudaMemcpyHostToDevice));
		CUDA_CHECK(cudaMemcpy(d_fwd, fwd_y, ysz, cudaMemcpyHostToDevice));
		CUDA_CHECK(cudaMemcpy(d_fwd + ysz, fwd_cr, csz, cudaMemcpyHostToDevice));
		CUDA_CHECK(cudaMemcpy(d_fwd + ysz + csz, fwd_cb, csz, cudaMemcpyHostToDevice));
		CUDA_CHECK(cudaMemcpy(d_cur, cur_y, ysz, cudaMemcpyHostToDevice));
		CUDA_CHECK(cudaMemcpy(d_cur + ysz, cur_cr, csz, cudaMemcpyHostToDevice));
		CUDA_CHECK(cudaMemcpy(d_cur + ysz + csz, cur_cb, csz, cudaMemcpyHostToDevice));
		ReconTask t{};
		t.hdr = d_hdr; t.coef = d_coef;
		t.cur = PlaneSet{d_cur, d_cur + ysz, d_cur + ysz + csz};
		t.fwd = PlaneSet{d_fwd, d_fwd + ysz, d_fwd + ysz + csz};
		t.mb_width = mb_width; t.mb_size = (int)n_mb;
		t.coded_width = mb_width * 16; t.coded_height = mb_height * 16;
		launch_reconstruct(&t, 1, 0);
		CUDA_CHECK(cudaGetLastError());
		CUDA_CHECK(cudaDeviceSynchronize());
		CUDA_CHECK(cudaMemcpy(cur_y, d_cur, ysz, cudaMemcpyDeviceToHost));
		CUDA_CHECK(cudaMemcpy(cur_cr, d_cur + ysz, csz, cudaMemcpyDeviceToHost));
		CUDA_CHECK(cudaMemcpy(cur_cb, d_cur + ysz + csz, csz, cudaMemcpyDeviceToHost));
		cudaFree(d_hdr); cudaFree(d_coef); cudaFree(d_fwd); cudaFree(d_cur);
		return 0;
	} catch (const std::exception &e) {
		fprintf(stderr, "%s\n", e.what());
		return -1;
	}
}

int jsmpeg_b200_debug_reconstruct_batch(int kind, int n_tasks, const int32_t *geometry, size_t cap_mb, size_t cap,
                                        size_t rgba_cap, void *const *hdr, void *const *coef, void *const *fwd,
                                        void *const *bwd, void *const *cur, void *const *rgba) {
	const bool is_b = kind == JSMPEG_B200_RECON_B || kind == JSMPEG_B200_RECON_RGBA_B;
	const bool is_rgba = kind == JSMPEG_B200_RECON_RGBA || kind == JSMPEG_B200_RECON_RGBA_B;
	if (kind < JSMPEG_B200_RECON_PLANES || kind > JSMPEG_B200_RECON_RGBA_B || n_tasks < 1) return -1;
	for (int i = 0; i < n_tasks; i++) {  // every buffer must hold what the task's own launch may touch
		const int32_t *g = geometry + 4 * i;
		const size_t mbw = g[0], mbh = g[1];
		if (g[0] < 1 || g[1] < 1 || mbw * mbh > cap_mb || mbw * mbh * 384 + mbw * 16 + 64 > cap) return -1;
		if (is_rgba && (g[2] < 1 || g[3] < 1 || (size_t)g[2] > mbw * 16 || (size_t)g[3] > mbh * 16 ||
		                (size_t)g[2] * g[3] * 4 > rgba_cap))
			return -1;
	}
	// one allocation per buffer, so that an access past a buffer is an access past an allocation
	std::vector<void *> allocs;
	auto alloc_copy = [&](const void *src, size_t bytes) {
		uint8_t *d = dev_alloc<uint8_t>(bytes);
		allocs.push_back(d);
		CUDA_CHECK(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
		return d;
	};
	int rc = 0;
	try {
		std::vector<ReconTask> tasks(n_tasks);
		std::vector<uint8_t *> d_bufs;  // per task: hdr, coef, fwd, bwd, cur, rgba (nullptr where unused)
		for (int i = 0; i < n_tasks; i++) {
			const int32_t *g = geometry + 4 * i;
			const size_t ysz = (size_t)g[0] * g[1] * 256, csz = ysz / 4;
			uint8_t *d_hdr = alloc_copy(hdr[i], cap_mb * sizeof(mb_record_t));
			uint8_t *d_coef = alloc_copy(coef[i], cap_mb * MB_COEF_INT16 * sizeof(int16_t));
			uint8_t *d_fwd = alloc_copy(fwd[i], cap);
			uint8_t *d_bwd = is_b ? alloc_copy(bwd[i], cap) : nullptr;
			uint8_t *d_cur = alloc_copy(cur[i], cap);
			uint8_t *d_rgba = is_rgba ? alloc_copy(rgba[i], rgba_cap) : nullptr;
			d_bufs.insert(d_bufs.end(), {d_hdr, d_coef, d_fwd, d_bwd, d_cur, d_rgba});
			ReconTask &t = tasks[i];
			t.hdr = reinterpret_cast<const mb_record_t *>(d_hdr);
			t.coef = reinterpret_cast<const int16_t *>(d_coef);
			t.cur = PlaneSet{d_cur, d_cur + ysz, d_cur + ysz + csz};
			t.fwd = PlaneSet{d_fwd, d_fwd + ysz, d_fwd + ysz + csz};
			if (is_b) t.bwd = PlaneSet{d_bwd, d_bwd + ysz, d_bwd + ysz + csz};
			t.mb_width = g[0]; t.mb_size = g[0] * g[1];
			t.coded_width = g[0] * 16; t.coded_height = g[1] * 16;
			t.rgba = d_rgba; t.width = g[2]; t.height = g[3];
		}
		// one call over all tasks: the launcher splits them into launches and sizes each grid as the engine's calls do
		if (kind == JSMPEG_B200_RECON_PLANES) launch_reconstruct(tasks.data(), n_tasks, 0);
		else if (kind == JSMPEG_B200_RECON_RGBA) launch_reconstruct_rgba(tasks.data(), n_tasks, 0);
		else launch_reconstruct_b(tasks.data(), n_tasks, is_rgba, 0);
		CUDA_CHECK(cudaGetLastError());
		CUDA_CHECK(cudaDeviceSynchronize());
		for (int i = 0; i < n_tasks; i++) {
			void *const host[6] = {hdr[i], coef[i], fwd[i], is_b ? bwd[i] : nullptr, cur[i], is_rgba ? rgba[i] : nullptr};
			const size_t bytes[6] = {cap_mb * sizeof(mb_record_t), cap_mb * MB_COEF_INT16 * sizeof(int16_t), cap, cap, cap, rgba_cap};
			for (int k = 0; k < 6; k++)
				if (host[k]) CUDA_CHECK(cudaMemcpy(host[k], d_bufs[6 * i + k], bytes[k], cudaMemcpyDeviceToHost));
		}
	} catch (const std::exception &e) {
		fprintf(stderr, "%s\n", e.what());
		rc = -1;
	}
	for (void *p : allocs) cudaFree(p);
	return rc;
}

}  // extern "C"

/* ORACLE — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement (plain C) of the arithmetic behind zarc's content path.  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use it.
 *
 * The reference (passcod/zarc) does not contain this arithmetic itself; it calls
 *   - crate blake3 1.5.0           (Cargo.lock:191-192)   at crates/zarc/src/encode/content_frame.rs:26,
 *                                                            crates/zarc/src/decode/frame_iterator.rs:77,99,
 *                                                            crates/zarc/src/integrity.rs:110
 *   - zstd-safe 7.0.0 -> zstd-sys 2.0.9+zstd.1.5.5 (Cargo.lock:2471-2481), i.e. libzstd 1.5.5
 *                                                        at crates/zarc/src/encode/lowlevel_frames.rs:30 (compress2)
 *                                                           crates/zarc/src/decode/zstd_iterator.rs:104-107,126-129
 * neither of which is vendored under /root/reference.  So this file restates the PUBLISHED
 * algorithms (BLAKE3 spec; RFC 8878 Zstandard frame format; XXH64 spec) and is pinned by
 * tests/test_oracle.py against (a) the libzstd.so.1.5.5 shipped in this image (the very version
 * zstd-sys vendors), (b) the Python `blake3` and `xxhash` packages, and (c) the known-answer
 * vectors of SURVEY.md App. B/E (tests/golden/).  The reference has no tests or golden vectors of
 * its own for this path (only crates/zarc-cli/src/args.rs:86-90), so "parity pinned by the
 * reference's own vectors" is impossible: PARITY IS PINNED TO THE SAME-VERSION THIRD-PARTY
 * LIBRARIES INSTEAD.
 *
 * The compressor is NOT restated: the reference's compressed bytes are exactly libzstd 1.5.5's
 * output, which oracle/ref_path.py obtains by dlopen()ing that library with the reference's call
 * sequence (encode.rs:61-62, content_frame.rs:37-39, lowlevel_frames.rs:21,30).
 */
#include <stdint.h>
#include <stddef.h>
#include <string.h>
#include <stdlib.h>

#define ZO_ERR(code) ((size_t)0 - (size_t)(code))
enum {
	ZO_E_GENERIC = 1,
	ZO_E_PREFIX = 10,        /* unknown frame magic */
	ZO_E_UNSUPPORTED = 14,   /* reserved bit / dictionary */
	ZO_E_CORRUPT = 20,
	ZO_E_CHECKSUM = 22,
	ZO_E_DST_SMALL = 70,
	ZO_E_SRC_SIZE = 72
};
int zo_is_error(size_t r) { return r > (size_t)-120; }

/* ======================================================================================
 * BLAKE3 (hash mode, 32-byte output).  blake3 crate call sites: content_frame.rs:26 etc.
 * ====================================================================================== */
static const uint32_t B3_IV[8] = {0x6A09E667, 0xBB67AE85, 0x3C6EF372, 0xA54FF53A,
                                  0x510E527F, 0x9B05688C, 0x1F83D9AB, 0x5BE0CD19};
static const uint8_t B3_PERM[16] = {2, 6, 3, 10, 7, 0, 4, 13, 1, 11, 12, 5, 9, 14, 15, 8};
enum { B3_CHUNK_START = 1, B3_CHUNK_END = 2, B3_PARENT = 4, B3_ROOT = 8 };

static uint32_t ror32(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }
static void b3_g(uint32_t* s, int a, int b, int c, int d, uint32_t mx, uint32_t my) {
	s[a] = s[a] + s[b] + mx; s[d] = ror32(s[d] ^ s[a], 16);
	s[c] = s[c] + s[d];      s[b] = ror32(s[b] ^ s[c], 12);
	s[a] = s[a] + s[b] + my; s[d] = ror32(s[d] ^ s[a], 8);
	s[c] = s[c] + s[d];      s[b] = ror32(s[b] ^ s[c], 7);
}
static void b3_compress(const uint32_t cv[8], const uint32_t block[16], uint64_t counter,
                        uint32_t block_len, uint32_t flags, uint32_t out_cv[8]) {
	uint32_t s[16], m[16], t[16];
	int i, r;
	for (i = 0; i < 8; i++) s[i] = cv[i];
	for (i = 0; i < 4; i++) s[8 + i] = B3_IV[i];
	s[12] = (uint32_t)counter; s[13] = (uint32_t)(counter >> 32); s[14] = block_len; s[15] = flags;
	memcpy(m, block, 64);
	for (r = 0; r < 7; r++) {
		b3_g(s, 0, 4, 8, 12, m[0], m[1]);   b3_g(s, 1, 5, 9, 13, m[2], m[3]);
		b3_g(s, 2, 6, 10, 14, m[4], m[5]);  b3_g(s, 3, 7, 11, 15, m[6], m[7]);
		b3_g(s, 0, 5, 10, 15, m[8], m[9]);  b3_g(s, 1, 6, 11, 12, m[10], m[11]);
		b3_g(s, 2, 7, 8, 13, m[12], m[13]); b3_g(s, 3, 4, 9, 14, m[14], m[15]);
		for (i = 0; i < 16; i++) t[i] = m[B3_PERM[i]];
		memcpy(m, t, 64);
	}
	for (i = 0; i < 8; i++) out_cv[i] = s[i] ^ s[i + 8];
}
static void b3_load_block(const uint8_t* p, size_t n, uint32_t w[16]) {
	uint8_t buf[64];
	int i;
	memset(buf, 0, 64);
	memcpy(buf, p, n);
	for (i = 0; i < 16; i++)
		w[i] = (uint32_t)buf[4 * i] | ((uint32_t)buf[4 * i + 1] << 8) | ((uint32_t)buf[4 * i + 2] << 16) |
		       ((uint32_t)buf[4 * i + 3] << 24);
}
/* chaining value of one chunk (<= 1024 bytes); root applies to the last block if is_root */
static void b3_chunk_cv(const uint8_t* p, size_t n, uint64_t chunk_idx, int is_root, uint32_t out[8]) {
	uint32_t cv[8], w[16];
	size_t nblocks = n == 0 ? 1 : (n + 63) / 64, b;
	memcpy(cv, B3_IV, 32);
	for (b = 0; b < nblocks; b++) {
		size_t off = b * 64, len = n - off > 64 ? 64 : n - off;
		uint32_t flags = (b == 0 ? B3_CHUNK_START : 0) | (b + 1 == nblocks ? B3_CHUNK_END : 0);
		if (b + 1 == nblocks && is_root) flags |= B3_ROOT;
		b3_load_block(p + off, len, w);
		b3_compress(cv, w, chunk_idx, (uint32_t)len, flags, cv);
	}
	memcpy(out, cv, 32);
}
static void b3_parent(const uint32_t l[8], const uint32_t r[8], int is_root, uint32_t out[8]) {
	uint32_t w[16];
	memcpy(w, l, 32);
	memcpy(w + 8, r, 32);
	b3_compress(B3_IV, w, 0, 64, B3_PARENT | (is_root ? B3_ROOT : 0), out);
}
/* recursive definition straight from the spec: left subtree = largest power of two < n chunks */
static void b3_subtree(const uint8_t* p, size_t n, uint64_t chunk0, int is_root, uint32_t out[8]) {
	if (n <= 1024) {
		b3_chunk_cv(p, n, chunk0, is_root, out);
		return;
	}
	{
		size_t chunks = (n + 1023) / 1024, left = 1;
		uint32_t l[8], r[8];
		while (left * 2 < chunks) left *= 2;
		b3_subtree(p, left * 1024, chunk0, 0, l);
		b3_subtree(p + left * 1024, n - left * 1024, chunk0 + left, 0, r);
		b3_parent(l, r, is_root, out);
	}
}
void zo_blake3(const uint8_t* data, size_t n, uint8_t out[32]) {
	uint32_t cv[8];
	int i;
	b3_subtree(data, n, 0, 1, cv);
	for (i = 0; i < 8; i++) {
		out[4 * i] = (uint8_t)cv[i]; out[4 * i + 1] = (uint8_t)(cv[i] >> 8);
		out[4 * i + 2] = (uint8_t)(cv[i] >> 16); out[4 * i + 3] = (uint8_t)(cv[i] >> 24);
	}
}

/* ======================================================================================
 * XXH64 (zstd Content_Checksum = low 32 bits, seed 0; RFC 8878 3.1.1)
 * ====================================================================================== */
#define XP1 0x9E3779B185EBCA87ULL
#define XP2 0xC2B2AE3D27D4EB4FULL
#define XP3 0x165667B19E3779F9ULL
#define XP4 0x85EBCA77C2B2AE63ULL
#define XP5 0x27D4EB2F165667C5ULL
static uint64_t rol64(uint64_t x, int n) { return (x << n) | (x >> (64 - n)); }
static uint64_t rd64(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }
static uint32_t rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
static uint64_t xround(uint64_t acc, uint64_t v) { return rol64(acc + v * XP2, 31) * XP1; }
uint64_t zo_xxh64(const uint8_t* p, size_t n, uint64_t seed) {
	const uint8_t* end = p + n;
	uint64_t h;
	if (n >= 32) {
		uint64_t v1 = seed + XP1 + XP2, v2 = seed + XP2, v3 = seed, v4 = seed - XP1;
		do {
			v1 = xround(v1, rd64(p)); v2 = xround(v2, rd64(p + 8));
			v3 = xround(v3, rd64(p + 16)); v4 = xround(v4, rd64(p + 24));
			p += 32;
		} while (p + 32 <= end);
		h = rol64(v1, 1) + rol64(v2, 7) + rol64(v3, 12) + rol64(v4, 18);
		h = (h ^ xround(0, v1)) * XP1 + XP4; h = (h ^ xround(0, v2)) * XP1 + XP4;
		h = (h ^ xround(0, v3)) * XP1 + XP4; h = (h ^ xround(0, v4)) * XP1 + XP4;
	} else {
		h = seed + XP5;
	}
	h += (uint64_t)n;
	while (p + 8 <= end) { h = rol64(h ^ xround(0, rd64(p)), 27) * XP1 + XP4; p += 8; }
	if (p + 4 <= end) { h = rol64(h ^ ((uint64_t)rd32(p) * XP1), 23) * XP2 + XP3; p += 4; }
	while (p < end) { h = rol64(h ^ ((uint64_t)*p * XP5), 11) * XP1; p++; }
	h ^= h >> 33; h *= XP2; h ^= h >> 29; h *= XP3; h ^= h >> 32;
	return h;
}

/* ======================================================================================
 * Zstandard frame decoder (RFC 8878).  Replaces DCtx::decompress_stream as used at
 * crates/zarc/src/decode/zstd_iterator.rs:104-107.
 * ====================================================================================== */
typedef struct { const uint8_t* p; int64_t bits; } zo_bits; /* backward stream: `bits` = unread bit count */

static int highbit(uint32_t v) { int r = -1; while (v) { v >>= 1; r++; } return r; }

/* read n (<=56) bits below the current position; bits before the start of the stream read as 0 */
static uint64_t bs_peek(const zo_bits* b, int n) {
	int64_t lo = b->bits - n; /* index of the lowest bit to read */
	uint64_t v = 0;
	int k;
	/* bit-by-bit gather: this is an oracle, clarity over speed */
	for (k = 0; k < n; k++) {
		int64_t bit = lo + k;
		if (bit >= 0) v |= (uint64_t)((b->p[bit >> 3] >> (bit & 7)) & 1) << k;
	}
	return v;
}
static uint64_t bs_read(zo_bits* b, int n) {
	uint64_t v = bs_peek(b, n);
	b->bits -= n;
	return v;
}
/* initialise from a byte range whose last byte carries the padding marker */
static int bs_init(zo_bits* b, const uint8_t* p, size_t n) {
	if (n == 0 || p[n - 1] == 0) return -1;
	b->p = p;
	b->bits = (int64_t)(n - 1) * 8 + highbit(p[n - 1]);
	return 0;
}

/* ---- FSE ---- */
typedef struct { uint8_t sym; uint8_t nb; uint16_t base; } zo_fse_e;
typedef struct { zo_fse_e e[512]; int log; } zo_fse_t;

/* forward bit reader for NCount */
static int fse_read_ncount(const uint8_t* src, size_t n, int max_log, int max_sym, int16_t* norm, int* nsym,
                           int* log_out, size_t* used) {
	uint64_t pos = 0; /* bit position */
	size_t nbits = n * 8;
	int log, remaining, sym = 0;
#define NC_READ(cnt, out)                                                       \
	do {                                                                        \
		uint32_t v_ = 0; int i_;                                                \
		if (pos + (cnt) > nbits) return -1;                                     \
		for (i_ = 0; i_ < (cnt); i_++) v_ |= (uint32_t)((src[(pos + i_) >> 3] >> ((pos + i_) & 7)) & 1) << i_; \
		pos += (cnt); (out) = v_;                                               \
	} while (0)
	uint32_t v;
	NC_READ(4, v);
	log = (int)v + 5;
	if (log > max_log) return -1;
	remaining = 1 << log;
	while (remaining > 0 && sym <= max_sym) {
		int bits = highbit((uint32_t)remaining + 1) + 1;
		uint32_t thr = (1u << bits) - 1 - ((uint32_t)remaining + 1);
		uint32_t val;
		int prob;
		NC_READ(bits - 1, val);
		if (val >= thr) { /* large value: one more bit; upper half is shifted down by thr */
			uint32_t hi;
			NC_READ(1, hi);
			val |= hi << (bits - 1);
			if (hi) val -= thr;
		}
		prob = (int)val - 1;
		norm[sym++] = (int16_t)prob;
		remaining -= prob < 0 ? 1 : prob;
		if (prob == 0) {
			uint32_t rep;
			do {
				int k;
				NC_READ(2, rep);
				for (k = 0; k < (int)rep; k++) { if (sym > max_sym) return -1; norm[sym++] = 0; }
			} while (rep == 3);
		}
	}
	if (remaining != 0 || sym > max_sym + 1) return -1;
	*nsym = sym; *log_out = log; *used = (size_t)((pos + 7) / 8);
	return 0;
#undef NC_READ
}
static void fse_build(zo_fse_t* t, const int16_t* norm, int nsym, int log) {
	int size = 1 << log, high = size - 1, s, i, pos = 0;
	int step = (size >> 1) + (size >> 3) + 3, mask = size - 1;
	uint16_t next[256];
	t->log = log;
	for (s = 0; s < nsym; s++) {
		if (norm[s] == -1) { t->e[high--].sym = (uint8_t)s; next[s] = 1; }
		else next[s] = (uint16_t)norm[s];
	}
	for (s = 0; s < nsym; s++)
		for (i = 0; i < norm[s]; i++) {
			t->e[pos].sym = (uint8_t)s;
			do { pos = (pos + step) & mask; } while (pos > high);
		}
	for (i = 0; i < size; i++) {
		uint16_t x = next[t->e[i].sym]++;
		int nb = log - highbit(x);
		t->e[i].nb = (uint8_t)nb;
		t->e[i].base = (uint16_t)((x << nb) - size);
	}
}
static void fse_build_rle(zo_fse_t* t, uint8_t sym) { t->log = 0; t->e[0].sym = sym; t->e[0].nb = 0; t->e[0].base = 0; }

/* statistics the tests use to make sure every format feature is covered */
typedef struct {
	uint64_t blocks_raw, blocks_rle, blocks_compressed;
	uint64_t lit_raw, lit_rle, lit_huf1, lit_huf4, lit_treeless;
	uint64_t seq_mode[4]; /* predefined, rle, fse, repeat (summed over LL/OF/ML) */
	uint64_t sequences, rep_offsets;
	uint64_t window_size, has_checksum, single_segment;
	/* ---- coverage of the encoder's edges (what a frame writer chose, not what the input was) ---- */
	uint64_t lit_fmt[4][4];          /* literals type (raw, rle, huffman, treeless) x Size_Format (0..3) */
	uint64_t huf_max_bits;           /* largest Huffman max_bits of a tree read */
	uint64_t huf_wdirect, huf_wfse;  /* Huffman weight descriptions: direct (4-bit) / FSE-compressed */
	uint64_t regen_max[4], regen_min[4]; /* Regenerated_Size extremes per literals type (min: ~0 while none seen) */
	uint64_t nseq_hdr[3];            /* Number_of_Sequences fields of 1 / 2 / 3 bytes (nseq = 0 counts as 1 byte) */
	uint64_t max_ll_code, max_ml_code, max_of_code;
	uint64_t tab_mode[3][4];         /* table (LL, OF, ML) x mode (predefined, rle, fse, repeat) */
	uint64_t max_log[3];             /* largest accuracy log of a table built per table (LL, OF, ML; RLE: 0) */
	uint64_t min_match, max_match;   /* over the resolved sequences (min: ~0 while none seen) */
	uint64_t max_offset;             /* after repeat codes are resolved */
	uint64_t max_lit_run;            /* largest Literals_Length of a sequence */
	uint64_t xblock_matches;         /* matches whose source starts before their block's first output byte */
	uint64_t xblock_reps;            /* repeat codes that resolve to an offset set in an earlier block */
	uint64_t fcs_size;               /* Frame_Content_Size field bytes: 0, 1, 2, 4 or 8 */
	uint64_t blocks;
	uint64_t huf_max_sym;            /* largest Huffman maxsym (the symbol whose weight is implied) */
	uint64_t huf_min_nw;             /* fewest explicit weights in a tree description (~0 while none seen) */
	uint64_t huf_max_nsym;           /* most symbols of non-zero weight in one tree */
} zo_stats;

#define ZO_MAX(a, b) ((a) = (a) > (uint64_t)(b) ? (a) : (uint64_t)(b))
#define ZO_MIN(a, b) ((a) = (a) < (uint64_t)(b) ? (a) : (uint64_t)(b))

/* ---- Huffman ---- */
typedef struct { uint8_t sym[2048]; uint8_t nb[2048]; int max_bits; int valid; } zo_huf_t;

static int huf_read_tree(zo_huf_t* h, const uint8_t* src, size_t n, size_t* used, zo_stats* st) {
	uint8_t w[256];
	int nw = 0, i;
	uint32_t sum = 0, left;
	int max_bits, last;
	uint32_t rank_count[13], rank_start[13];
	if (n < 1) return -1;
	if (src[0] >= 128) {
		nw = src[0] - 127;
		if (1 + (size_t)(nw + 1) / 2 > n) return -1;
		for (i = 0; i < nw; i++) w[i] = (i & 1) ? (src[1 + i / 2] & 15) : (src[1 + i / 2] >> 4);
		*used = 1 + (size_t)(nw + 1) / 2;
	} else {
		size_t csz = src[0], nc_used;
		int16_t norm[256];
		int nsym, log;
		zo_fse_t t;
		zo_bits b;
		uint32_t s1, s2;
		if (1 + csz > n || csz < 2) return -1;
		if (fse_read_ncount(src + 1, csz, 6, 255, norm, &nsym, &log, &nc_used)) return -1;
		if (nc_used >= csz) return -1;
		fse_build(&t, norm, nsym, log);
		if (bs_init(&b, src + 1 + nc_used, csz - nc_used)) return -1;
		s1 = (uint32_t)bs_read(&b, log);
		s2 = (uint32_t)bs_read(&b, log);
		for (;;) {
			if (nw > 253) return -1;
			w[nw++] = t.e[s1].sym;
			s1 = t.e[s1].base + (uint32_t)bs_read(&b, t.e[s1].nb);
			if (b.bits < 0) { w[nw++] = t.e[s2].sym; break; }
			w[nw++] = t.e[s2].sym;
			s2 = t.e[s2].base + (uint32_t)bs_read(&b, t.e[s2].nb);
			if (b.bits < 0) { w[nw++] = t.e[s1].sym; break; }
		}
		*used = 1 + csz;
	}
	for (i = 0; i < nw; i++) { if (w[i] > 11) return -1; if (w[i]) sum += 1u << (w[i] - 1); }
	if (sum == 0) return -1;
	max_bits = highbit(sum) + 1;
	if (max_bits > 11) return -1;
	left = (1u << max_bits) - sum;
	if (left & (left - 1)) return -1; /* must be a power of two */
	last = highbit(left) + 1;
	w[nw++] = (uint8_t)last;
	memset(rank_count, 0, sizeof rank_count);
	for (i = 0; i < nw; i++) rank_count[w[i]]++;
	if (rank_count[1] < 2 || (rank_count[1] & 1)) return -1; /* as libzstd HUF_readStats */
	rank_start[1] = 0;
	for (i = 1; i < 12; i++) rank_start[i + 1] = rank_start[i] + (rank_count[i] << (i - 1));
	for (i = 0; i < nw; i++)
		if (w[i]) {
			uint32_t len = 1u << (w[i] - 1), k;
			for (k = 0; k < len; k++) {
				h->sym[rank_start[w[i]] + k] = (uint8_t)i;
				h->nb[rank_start[w[i]] + k] = (uint8_t)(max_bits + 1 - w[i]);
			}
			rank_start[w[i]] += len;
		}
	h->max_bits = max_bits;
	h->valid = 1;
	if (st) {
		ZO_MAX(st->huf_max_bits, max_bits);
		if (src[0] >= 128) st->huf_wdirect++;
		else st->huf_wfse++;
		ZO_MAX(st->huf_max_sym, nw - 1);
		ZO_MIN(st->huf_min_nw, nw - 1);
		ZO_MAX(st->huf_max_nsym, nw - rank_count[0]);
	}
	return 0;
}
static int huf_decode_stream(const zo_huf_t* h, const uint8_t* src, size_t n, uint8_t* dst, size_t count) {
	zo_bits b;
	size_t i;
	if (bs_init(&b, src, n)) return -1;
	for (i = 0; i < count; i++) {
		uint32_t idx;
		if (b.bits >= h->max_bits) idx = (uint32_t)bs_peek(&b, h->max_bits);
		else idx = (uint32_t)(bs_peek(&b, (int)(b.bits < 0 ? 0 : b.bits)) << (h->max_bits - (b.bits < 0 ? 0 : b.bits)));
		dst[i] = h->sym[idx];
		b.bits -= h->nb[idx];
		if (b.bits < 0) return -1;
	}
	return b.bits == 0 ? 0 : -1;
}

/* ---- sequence code tables (RFC 8878 3.1.1.3.2.1.1) ---- */
static const uint32_t LL_BASE[36] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40,
                                     48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536};
static const uint8_t LL_BITS[36] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3,
                                    4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
static const uint32_t ML_BASE[53] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28,
                                     29, 30, 31, 32, 33, 34, 35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051,
                                     4099, 8195, 16387, 32771, 65539};
static const uint8_t ML_BITS[53] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                                    0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
static const int16_t LL_DEFAULT[36] = {4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1};
static const int16_t ML_DEFAULT[53] = {1, 4, 3, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,
                                       1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1, -1, -1};
static const int16_t OF_DEFAULT[29] = {1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1};

typedef struct {
	zo_huf_t huf;
	zo_fse_t ll, of, ml;
	int have_ll, have_of, have_ml;
	uint64_t rep[3];
	uint64_t rep_blk[3]; /* block in which each repeat slot's offset was set (the initial 1 / 4 / 8: block 0) */
	uint64_t blk;        /* index of the block being decoded */
} zo_frame_state;

static int seq_table(zo_fse_t* t, int* have, int which, int mode, const uint8_t** pp, const uint8_t* end, int max_log, int max_sym,
                     const int16_t* def, int def_n, int def_log, zo_stats* st) {
	if (st) { st->seq_mode[mode]++; st->tab_mode[which][mode]++; }
	switch (mode) {
	case 0: fse_build(t, def, def_n, def_log); *have = 1; if (st) ZO_MAX(st->max_log[which], def_log); return 0;
	case 1:
		if (*pp >= end) return -1;
		if (**pp > max_sym) return -1;
		fse_build_rle(t, **pp); (*pp)++; *have = 1; return 0;
	case 2: {
		int16_t norm[64];
		int nsym, log;
		size_t used;
		if (fse_read_ncount(*pp, (size_t)(end - *pp), max_log, max_sym, norm, &nsym, &log, &used)) return -1;
		fse_build(t, norm, nsym, log);
		if (st) ZO_MAX(st->max_log[which], log);
		*pp += used; *have = 1; return 0;
	}
	default: return *have ? 0 : -1;
	}
}

/* decode one Compressed block; dst0 = start of frame output (for back-references) */
static size_t decode_compressed_block(zo_frame_state* fs, const uint8_t* src, size_t n, uint8_t* dst0, size_t dpos,
                                      size_t dcap, uint64_t window, uint8_t* litbuf, zo_stats* st) {
	const uint8_t* p = src;
	const uint8_t* end = src + n;
	const uint8_t* lit;
	size_t regen, comp = 0, hdr;
	int ltype, sf, streams = 1;
	size_t out = dpos;
	if (n < 1) return ZO_ERR(ZO_E_CORRUPT);
	ltype = p[0] & 3; sf = (p[0] >> 2) & 3;
	if (ltype < 2) {
		if (sf == 0 || sf == 2) { regen = p[0] >> 3; hdr = 1; }
		else if (sf == 1) { if (n < 2) return ZO_ERR(ZO_E_CORRUPT); regen = (p[0] >> 4) | ((size_t)p[1] << 4); hdr = 2; }
		else { if (n < 3) return ZO_ERR(ZO_E_CORRUPT); regen = (p[0] >> 4) | ((size_t)p[1] << 4) | ((size_t)p[2] << 12); hdr = 3; }
		p += hdr;
		if (regen > 131072) return ZO_ERR(ZO_E_CORRUPT);
		if (ltype == 0) {
			if ((size_t)(end - p) < regen) return ZO_ERR(ZO_E_CORRUPT);
			lit = p; p += regen;
			if (st) st->lit_raw++;
		} else {
			if (p >= end) return ZO_ERR(ZO_E_CORRUPT);
			memset(litbuf, *p, regen); lit = litbuf; p++;
			if (st) st->lit_rle++;
		}
	} else {
		uint64_t v;
		if (n < 3) return ZO_ERR(ZO_E_CORRUPT);
		if (sf == 0 || sf == 1) { v = p[0] | (p[1] << 8) | ((uint64_t)p[2] << 16); regen = (v >> 4) & 1023; comp = (v >> 14) & 1023; hdr = 3; streams = sf == 0 ? 1 : 4; }
		else if (sf == 2) { if (n < 4) return ZO_ERR(ZO_E_CORRUPT); v = p[0] | (p[1] << 8) | ((uint64_t)p[2] << 16) | ((uint64_t)p[3] << 24); regen = (v >> 4) & 16383; comp = (v >> 18) & 16383; hdr = 4; streams = 4; }
		else { if (n < 5) return ZO_ERR(ZO_E_CORRUPT); v = p[0] | (p[1] << 8) | ((uint64_t)p[2] << 16) | ((uint64_t)p[3] << 24) | ((uint64_t)p[4] << 32); regen = (v >> 4) & 262143; comp = (v >> 22) & 262143; hdr = 5; streams = 4; }
		p += hdr;
		if (regen > 131072 || (size_t)(end - p) < comp) return ZO_ERR(ZO_E_CORRUPT);
		{
			const uint8_t* lp = p;
			const uint8_t* lend = p + comp;
			if (ltype == 2) {
				size_t used;
				if (huf_read_tree(&fs->huf, lp, comp, &used, st)) return ZO_ERR(ZO_E_CORRUPT);
				lp += used;
			} else {
				if (!fs->huf.valid) return ZO_ERR(ZO_E_CORRUPT);
				if (st) st->lit_treeless++;
			}
			if (streams == 1) {
				if (huf_decode_stream(&fs->huf, lp, (size_t)(lend - lp), litbuf, regen)) return ZO_ERR(ZO_E_CORRUPT);
				if (st && ltype == 2) st->lit_huf1++;
			} else {
				size_t s1, s2, s3, seg = (regen + 3) / 4;
				if (lend - lp < 6) return ZO_ERR(ZO_E_CORRUPT);
				s1 = lp[0] | (lp[1] << 8); s2 = lp[2] | (lp[3] << 8); s3 = lp[4] | (lp[5] << 8);
				lp += 6;
				if (s1 + s2 + s3 > (size_t)(lend - lp) || seg * 3 > regen) return ZO_ERR(ZO_E_CORRUPT);
				if (huf_decode_stream(&fs->huf, lp, s1, litbuf, seg)) return ZO_ERR(ZO_E_CORRUPT);
				if (huf_decode_stream(&fs->huf, lp + s1, s2, litbuf + seg, seg)) return ZO_ERR(ZO_E_CORRUPT);
				if (huf_decode_stream(&fs->huf, lp + s1 + s2, s3, litbuf + 2 * seg, seg)) return ZO_ERR(ZO_E_CORRUPT);
				if (huf_decode_stream(&fs->huf, lp + s1 + s2 + s3, (size_t)(lend - lp) - s1 - s2 - s3, litbuf + 3 * seg, regen - 3 * seg)) return ZO_ERR(ZO_E_CORRUPT);
				if (st && ltype == 2) st->lit_huf4++;
			}
			lit = litbuf;
			p = lend;
		}
	}
	if (st) {
		st->lit_fmt[ltype][sf]++;
		ZO_MAX(st->regen_max[ltype], regen);
		ZO_MIN(st->regen_min[ltype], regen);
	}
	/* sequences section */
	{
		uint32_t nseq;
		size_t lpos = 0;
		if (p >= end) return ZO_ERR(ZO_E_CORRUPT);
		/* the field length the frame used (a count below 128 may also be written in 2 bytes, one below 0x7F00 in 3) */
		if (st) st->nseq_hdr[p[0] < 128 ? 0 : p[0] < 255 ? 1 : 2]++;
		if (p[0] == 0) { nseq = 0; p++; }
		else if (p[0] < 128) { nseq = p[0]; p++; }
		else if (p[0] < 255) { if (end - p < 2) return ZO_ERR(ZO_E_CORRUPT); nseq = ((uint32_t)(p[0] - 128) << 8) + p[1]; p += 2; }
		else { if (end - p < 3) return ZO_ERR(ZO_E_CORRUPT); nseq = p[1] + ((uint32_t)p[2] << 8) + 0x7F00; p += 3; }
		if (nseq) {
			int modes;
			zo_bits b;
			uint32_t sl, so, sm, i;
			if (p >= end) return ZO_ERR(ZO_E_CORRUPT);
			modes = *p++;
			if (modes & 3) return ZO_ERR(ZO_E_CORRUPT);
			if (seq_table(&fs->ll, &fs->have_ll, 0, (modes >> 6) & 3, &p, end, 9, 35, LL_DEFAULT, 36, 6, st)) return ZO_ERR(ZO_E_CORRUPT);
			if (seq_table(&fs->of, &fs->have_of, 1, (modes >> 4) & 3, &p, end, 8, 31, OF_DEFAULT, 29, 5, st)) return ZO_ERR(ZO_E_CORRUPT);
			if (seq_table(&fs->ml, &fs->have_ml, 2, (modes >> 2) & 3, &p, end, 9, 52, ML_DEFAULT, 53, 6, st)) return ZO_ERR(ZO_E_CORRUPT);
			if (bs_init(&b, p, (size_t)(end - p))) return ZO_ERR(ZO_E_CORRUPT);
			sl = (uint32_t)bs_read(&b, fs->ll.log);
			so = (uint32_t)bs_read(&b, fs->of.log);
			sm = (uint32_t)bs_read(&b, fs->ml.log);
			if (b.bits < 0) return ZO_ERR(ZO_E_CORRUPT);
			for (i = 0; i < nseq; i++) {
				uint32_t oc = fs->of.e[so].sym, mc = fs->ml.e[sm].sym, lc = fs->ll.e[sl].sym;
				uint64_t ov, offset;
				uint32_t ml, ll;
				if (oc > 31 || mc > 52 || lc > 35) return ZO_ERR(ZO_E_CORRUPT);
				if (st) { ZO_MAX(st->max_ll_code, lc); ZO_MAX(st->max_ml_code, mc); ZO_MAX(st->max_of_code, oc); }
				ov = ((uint64_t)1 << oc) + bs_read(&b, (int)oc);
				ml = ML_BASE[mc] + (uint32_t)bs_read(&b, ML_BITS[mc]);
				ll = LL_BASE[lc] + (uint32_t)bs_read(&b, LL_BITS[lc]);
				if (i + 1 < nseq) {
					sl = fs->ll.e[sl].base + (uint32_t)bs_read(&b, fs->ll.e[sl].nb);
					sm = fs->ml.e[sm].base + (uint32_t)bs_read(&b, fs->ml.e[sm].nb);
					so = fs->of.e[so].base + (uint32_t)bs_read(&b, fs->of.e[so].nb);
				}
				if (b.bits < 0) return ZO_ERR(ZO_E_CORRUPT);
				/* repeat-offset resolution */
				if (ov > 3) {
					offset = ov - 3;
					fs->rep[2] = fs->rep[1]; fs->rep[1] = fs->rep[0]; fs->rep[0] = offset;
					fs->rep_blk[2] = fs->rep_blk[1]; fs->rep_blk[1] = fs->rep_blk[0]; fs->rep_blk[0] = fs->blk;
				} else {
					uint32_t idx = (uint32_t)ov - 1 + (ll == 0 ? 1 : 0);
					uint64_t from; /* the block the resolved offset was set in (it keeps that as it moves between slots) */
					if (st) st->rep_offsets++;
					if (idx == 0) { offset = fs->rep[0]; from = fs->rep_blk[0]; }
					else {
						offset = idx == 3 ? fs->rep[0] - 1 : fs->rep[idx];
						from = fs->rep_blk[idx == 3 ? 0 : idx];
						if (offset == 0) return ZO_ERR(ZO_E_CORRUPT);
						if (idx > 1) { fs->rep[2] = fs->rep[1]; fs->rep_blk[2] = fs->rep_blk[1]; }
						fs->rep[1] = fs->rep[0]; fs->rep_blk[1] = fs->rep_blk[0];
						fs->rep[0] = offset; fs->rep_blk[0] = from;
					}
					if (st && from < fs->blk) st->xblock_reps++;
				}
				if (st) {
					ZO_MIN(st->min_match, ml); ZO_MAX(st->max_match, ml);
					ZO_MAX(st->max_offset, offset); ZO_MAX(st->max_lit_run, ll);
				}
				/* execute */
				if (lpos + ll > regen) return ZO_ERR(ZO_E_CORRUPT);
				if (out + ll + ml > dcap) return ZO_ERR(ZO_E_DST_SMALL);
				memcpy(dst0 + out, lit + lpos, ll);
				out += ll; lpos += ll;
				if (offset > out || offset > window) return ZO_ERR(ZO_E_CORRUPT);
				if (st && out - offset < dpos) st->xblock_matches++;
				{
					uint32_t k;
					for (k = 0; k < ml; k++) dst0[out + k] = dst0[out + k - offset];
				}
				out += ml;
			}
			if (b.bits != 0) return ZO_ERR(ZO_E_CORRUPT);
			if (st) st->sequences += nseq;
		} else if (p != end) return ZO_ERR(ZO_E_CORRUPT);
		if (out + (regen - lpos) > dcap) return ZO_ERR(ZO_E_DST_SMALL);
		memcpy(dst0 + out, lit + lpos, regen - lpos);
		out += regen - lpos;
	}
	if (out - dpos > 131072) return ZO_ERR(ZO_E_CORRUPT);
	return out - dpos;
}

/* Decode exactly one Zstandard frame at src.  Returns bytes written or an error; *consumed = frame length. */
size_t zo_zstd_decompress_frame(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, size_t* consumed, zo_stats* st) {
	const uint8_t* p = src;
	const uint8_t* end = src + n;
	uint8_t desc;
	int fcs_flag, single, checksum, did_flag, fcs_len;
	uint64_t window = 0, fcs = 0;
	int have_fcs;
	size_t out = 0;
	zo_frame_state* fs;
	uint8_t* litbuf;
	size_t rc = 0;
	if (st) {
		memset(st, 0, sizeof *st);
		memset(st->regen_min, 0xff, sizeof st->regen_min);
		st->min_match = ~(uint64_t)0;
		st->huf_min_nw = ~(uint64_t)0;
	}
	if (n < 6) return ZO_ERR(ZO_E_SRC_SIZE);
	if (rd32(p) != 0xFD2FB528u) return ZO_ERR(ZO_E_PREFIX);
	desc = p[4]; p += 5;
	fcs_flag = desc >> 6; single = (desc >> 5) & 1; checksum = (desc >> 2) & 1; did_flag = desc & 3;
	if (desc & 8) return ZO_ERR(ZO_E_UNSUPPORTED);
	if (!single) {
		int wl;
		if (p >= end) return ZO_ERR(ZO_E_SRC_SIZE);
		wl = 10 + (*p >> 3);
		window = ((uint64_t)1 << wl) + (((uint64_t)1 << wl) >> 3) * (*p & 7);
		p++;
	}
	if (did_flag) {
		static const int dl[4] = {0, 1, 2, 4};
		uint32_t did = 0; int i;
		if (end - p < dl[did_flag]) return ZO_ERR(ZO_E_SRC_SIZE);
		for (i = 0; i < dl[did_flag]; i++) did |= (uint32_t)p[i] << (8 * i);
		p += dl[did_flag];
		if (did) return ZO_ERR(ZO_E_UNSUPPORTED);
	}
	fcs_len = fcs_flag == 0 ? (single ? 1 : 0) : fcs_flag == 1 ? 2 : fcs_flag == 2 ? 4 : 8;
	have_fcs = fcs_len != 0;
	if (end - p < fcs_len) return ZO_ERR(ZO_E_SRC_SIZE);
	{ int i; for (i = 0; i < fcs_len; i++) fcs |= (uint64_t)p[i] << (8 * i); }
	if (fcs_len == 2) fcs += 256;
	p += fcs_len;
	if (single) window = fcs;
	if (st) {
		st->window_size = window; st->has_checksum = (uint64_t)checksum; st->single_segment = (uint64_t)single;
		st->fcs_size = (uint64_t)fcs_len;
	}
	fs = (zo_frame_state*)calloc(1, sizeof *fs);
	litbuf = (uint8_t*)malloc(131072 + 32);
	fs->rep[0] = 1; fs->rep[1] = 4; fs->rep[2] = 8;
	for (;;) {
		uint32_t bh, bsize;
		int last, type;
		if (end - p < 3) { rc = ZO_ERR(ZO_E_SRC_SIZE); goto done; }
		bh = p[0] | (p[1] << 8) | ((uint32_t)p[2] << 16);
		p += 3;
		last = bh & 1; type = (bh >> 1) & 3; bsize = bh >> 3;
		if (type == 3 || bsize > 131072) { rc = ZO_ERR(ZO_E_CORRUPT); goto done; }
		if (type == 0) {
			if ((size_t)(end - p) < bsize) { rc = ZO_ERR(ZO_E_SRC_SIZE); goto done; }
			if (out + bsize > cap) { rc = ZO_ERR(ZO_E_DST_SMALL); goto done; }
			memcpy(dst + out, p, bsize); out += bsize; p += bsize;
			if (st) st->blocks_raw++;
		} else if (type == 1) {
			if (end - p < 1) { rc = ZO_ERR(ZO_E_SRC_SIZE); goto done; }
			if (out + bsize > cap) { rc = ZO_ERR(ZO_E_DST_SMALL); goto done; }
			memset(dst + out, *p, bsize); out += bsize; p++;
			if (st) st->blocks_rle++;
		} else {
			size_t r;
			if ((size_t)(end - p) < bsize) { rc = ZO_ERR(ZO_E_SRC_SIZE); goto done; }
			r = decode_compressed_block(fs, p, bsize, dst, out, cap, window ? window : (uint64_t)-1, litbuf, st);
			if (zo_is_error(r)) { rc = r; goto done; }
			out += r; p += bsize;
			if (st) st->blocks_compressed++;
		}
		if (st) st->blocks++;
		fs->blk++;
		if (last) break;
	}
	if (checksum) {
		if (end - p < 4) { rc = ZO_ERR(ZO_E_SRC_SIZE); goto done; }
		if (rd32(p) != (uint32_t)zo_xxh64(dst, out, 0)) { rc = ZO_ERR(ZO_E_CHECKSUM); goto done; }
		p += 4;
	}
	if (have_fcs && fcs != out) { rc = ZO_ERR(ZO_E_CORRUPT); goto done; }
	if (consumed) *consumed = (size_t)(p - src);
	rc = out;
done:
	free(fs);
	free(litbuf);
	return rc;
}

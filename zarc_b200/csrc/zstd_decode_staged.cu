// K5 + K6 for MULTI-BLOCK frames: the staged pipeline.  Replaces DCtx::decompress_stream as driven by
// crates/zarc/src/decode/zstd_iterator.rs:88-153 for frames of two blocks and more -- every content file above
// 128 KiB, whoever wrote it.
//
// A Zstandard frame is a serial chain of blocks for a streaming decoder: a block may re-use the previous block's
// Huffman tree (Treeless literals) and FSE tables (Repeat_Mode), starts from the previous block's repeat-offset
// history, and its matches reach back across block boundaries up to the window.  libzstd writes all of these at
// levels 1/3/9 (SURVEY.md App. E).  Decoding such a frame block after block with one warp runs at 15-50 MB/s; here
// the work is staged so that everything except the copies themselves is parallel over ALL blocks of ALL frames:
//
//   1. walk     (thread per frame)  block headers -> one descriptor per block               [k_zds_count, k_zds_emit]
//   2. modes    (thread per block)  literals / sequences section headers: types, modes, counts          [k_zds_modes]
//   3. sources  (thread per frame)  "last block that defined it" for the Huffman tree and the LL / OF / ML tables:
//                                   a Treeless / Repeat_Mode block reads the description out of THAT block [k_zds_sources]
//   4. entropy  (warp per batch of blocks, one block per lane for the FSE streams) tables, Huffman literals and all
//               sequences of every block, into staging.  Offsets are kept SYMBOLIC where they come out of the repeat
//               history the block starts with (unknown yet): slot s minus k is stored as 2^27 + (s+1) 2^25 - k, a range
//               no real offset can take (windows are <= 2^27).  The same arithmetic the concrete history uses
//               ("rep0 - 1") works on these values unchanged; the history a block ends with is, likewise, three values
//               that are either concrete or "incoming slot s minus k": the block's TRANSFORMER.                [k_zds_entropy]
//   5. scan     (thread per frame)  output offset of every block (prefix sum of regenerated sizes) and the concrete
//               history every block starts with (transformers composed in block order)                   [k_zds_frame_scan]
//   6. execute  (warp per block, blocks handed out in block order) literal and match copies.  A block whose matches
//               stay inside it runs at once; a block that reads earlier output waits for exactly the blocks it reads
//               (release/acquire on per-block flags), so independent blocks (this library's encoder) all run in
//               parallel and dependent ones (libzstd) run as a chain per frame, all frames at once.              [k_zds_exec]
//
// Steps 4-6 run over chunks of blocks (the same range of block indices of every frame, so that all frames advance
// together) to bound the staging memory.  Bytes, per-frame status codes and checksum handling equal the serial decoder's.
#include "common.h"
#include "zstd_common.cuh"
#include "zstd_decode.cuh"
#include "xxh64.cuh"
#include <vector>

#define ZDS_NONE 0xffffffffu
#define ZDS_MAXSEQ 43691u               // a block regenerates <= 128 KiB and every sequence >= 3 bytes
#define ZDS_WIN_MAX (1u << 27)          // largest window (and so offset) the decoder accepts (zd_frame_header)
#define ZDS_HMAX (1u << 20)             // frames of more blocks than this are left to the serial path (128 GiB)
#define ZDS_CHUNK_ITEMS 32768u          // blocks per chunk (<= 4 GiB of output)
#define ZDS_CHUNK_WIDTH 4096u           // block indices per chunk at most
#define ZDS_WARPS 4
#define ZDS_ENT_CTAS 5
#define ZDS_EXEC_CTAS 6

// info word of a block
#define ZDS_I_LTYPE 3u       // Literals_Block_Type (compressed blocks)
#define ZDS_I_BAD 4u         // malformed block or section headers
#define ZDS_I_SEQ 8u         // Number_of_Sequences > 0
#define ZDS_I_MODES(i) (((i) >> 8) & 0xffu)   // Symbol_Compression_Modes byte
// result flags
#define ZDS_R_SYM 1u         // a match used an offset out of the incoming repeat history

struct ZdsBlk {      // per block of a staged frame; index g = first[k] + j
	u64 ip;          // offset of the 3-byte block header inside the frame
	u32 k, j;
	u32 hdr;         // Block_Header: last | type << 1 | size << 3
	u32 info;
	u32 nseq;
	u32 lit_regen;   // compressed blocks: Regenerated_Size of the literals section
	u32 src[4];      // block (index g) whose section describes the table in use: Huffman, LL, OF, ML
};
struct ZdsRes {      // what the entropy stage learned about a block
	u32 status;
	u32 regen;       // bytes the block regenerates
	u32 rep[3];      // repeat history after the block; symbolic entries refer to the history before it
	u32 need_back;   // how far before the block's first byte its matches with concrete offsets reach
	u32 flags;
	u32 lit_used;    // literals consumed by the sequences (the rest follows the last sequence)
};

ZG_DEV u32 zds_sym(u32 slot) { return ZDS_WIN_MAX + ((slot + 1u) << 25); }
ZG_DEV bool zds_is_sym(u32 off) { return off > ZDS_WIN_MAX; }
// symbolic value -> concrete, given the history it refers to; 0 when it would not be a valid offset
ZG_DEV u32 zds_resolve(u32 v, u32 r0, u32 r1, u32 r2) {
	if (!zds_is_sym(v)) return v;
	u32 slot = (v - ZDS_WIN_MAX - 1u) >> 25;
	u32 k = zds_sym(slot) - v;
	u32 r = slot == 0 ? r0 : slot == 1 ? r1 : r2;
	return r > k ? r - k : 0u;
}

// ---------------------------------------------------------------------------------------------
// 1. walk.  Which frames are staged: two blocks and more, well-formed headers, inside the archive and the output.
ZG_DEV u64 zds_walk(const u8* archive, u64 archive_len, u64 fo, u64 fl, u64 ul, u64 oo, u64 out_cap, u64 split_min, u32 k, ZdsBlk* blk,
                    u64* tail) {
	if (ul < split_min || fo > archive_len || fl > archive_len - fo || oo > out_cap || ul > out_cap - oo) return 0;
	ZdLane L;
	L.src = archive + fo;
	L.n = fl;
	L.status = ZS_OK;
	L.flags = 0;
	L.ip = L.fcs = 0;
	L.fcs_len = 0;
	zd_frame_header(L);
	if (L.status != ZS_OK || (L.fcs_len && L.fcs != ul)) return 0;
	u64 ip = L.ip, nb = 0;
	for (;;) {
		if (ip + 3 > fl) return 0;
		u32 bh = zg_ld24(L.src + ip);
		u32 last = bh & 1, type = (bh >> 1) & 3, bsize = bh >> 3;
		if (type == 3 || bsize > ZS_BLOCK_MAX) return 0;
		u64 body = type == 1 ? 1 : bsize;
		if (ip + 3 + body > fl) return 0;
		if (blk) {
			ZdsBlk& B = blk[nb];
			B.ip = ip;
			B.k = k;
			B.j = (u32)nb;
			B.hdr = bh;
		}
		nb++;
		ip += 3 + body;
		if (last) break;
		if (nb > ZDS_HMAX) return 0;
	}
	if (nb < 2) return 0;
	if (tail) *tail = ip;
	return nb;
}
// tot: [0] staged frames, [1] their blocks, [2] most blocks in one frame, [3] other frames
__global__ void __launch_bounds__(128)
k_zds_count(const u8* __restrict__ archive, u64 archive_len, const u64* __restrict__ off, const u64* __restrict__ len,
            const u64* __restrict__ ulen, const u64* __restrict__ out_off, u64 out_cap, u64 n, u64 split_min, u32* __restrict__ nblk,
            u64* __restrict__ first, u32* __restrict__ multi, u32* __restrict__ single, unsigned long long* tot, u32* __restrict__ hist) {
	u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= n) return;
	u64 nb = zds_walk(archive, archive_len, off[k], len[k], ulen[k], out_off[k], out_cap, split_min, (u32)k, nullptr, nullptr);
	nblk[k] = (u32)nb;
	if (nb) {
		multi[atomicAdd(&tot[0], 1ull)] = (u32)k;
		first[k] = atomicAdd(&tot[1], (unsigned long long)nb);
		atomicMax(&tot[2], (unsigned long long)nb);
		atomicAdd(&hist[nb], 1u);
	} else {
		single[atomicAdd(&tot[3], 1ull)] = (u32)k;
	}
}
__global__ void __launch_bounds__(128)
k_zds_emit(const u8* __restrict__ archive, u64 archive_len, const u64* __restrict__ off, const u64* __restrict__ len,
           const u64* __restrict__ ulen, const u64* __restrict__ out_off, u64 out_cap, const u32* __restrict__ multi, u64 nmulti, u64 split_min,
           const u64* __restrict__ first, ZdsBlk* __restrict__ blk, u64* __restrict__ tail, u64* __restrict__ f_out, u32* __restrict__ f_rep,
           u32* __restrict__ f_status, u32* __restrict__ done_upto) {
	u64 m = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (m >= nmulti) return;
	u32 k = multi[m];
	zds_walk(archive, archive_len, off[k], len[k], ulen[k], out_off[k], out_cap, split_min, k, blk + first[k], &tail[k]);
	f_out[k] = 0;
	f_rep[3 * (u64)k] = 1;  // the format's initial history (RFC 8878 3.1.1.5)
	f_rep[3 * (u64)k + 1] = 4;
	f_rep[3 * (u64)k + 2] = 8;
	f_status[k] = ZS_OK;
	done_upto[k] = 0;
}

// ---------------------------------------------------------------------------------------------
// 2. section headers of one compressed block (single thread).  Returns false when malformed.
struct ZdsSect {
	ZdLitHdr h;
	u32 nseq, modes;
	const u8* tables;   // first table description (after the modes byte)
};
ZG_DEV bool zds_sections(const u8* src, u32 n, ZdsSect& S) {
	if (!zd_lit_header(src, n, S.h)) return false;
	const u8* end = src + n;
	const u8* p = src + S.h.hdr + S.h.comp;
	if (p >= end) return false;
	u32 c0 = p[0];
	if (c0 < 128) {
		S.nseq = c0;
		p += 1;
	} else if (c0 < 255) {
		if (end - p < 2) return false;
		S.nseq = ((c0 - 128) << 8) + p[1];
		p += 2;
	} else {
		if (end - p < 3) return false;
		S.nseq = (u32)p[1] + ((u32)p[2] << 8) + 0x7F00;
		p += 3;
	}
	S.modes = 0;
	if (S.nseq == 0) {
		S.tables = p;
		return p == end;
	}
	if (p >= end) return false;
	S.modes = *p++;
	S.tables = p;
	return (S.modes & 3) == 0 && S.nseq <= ZDS_MAXSEQ;
}
__global__ void __launch_bounds__(128)
k_zds_modes(const u8* __restrict__ archive, const u64* __restrict__ off, ZdsBlk* __restrict__ blk, u64 nblocks) {
	u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (g >= nblocks) return;
	ZdsBlk B = blk[g];
	u32 type = (B.hdr >> 1) & 3, bsize = B.hdr >> 3;
	u32 info = 0, nseq = 0, regen = 0;
	if (type == 2) {
		ZdsSect S;
		if (bsize == 0 || !zds_sections(archive + off[B.k] + B.ip + 3, bsize, S)) info = ZDS_I_BAD;
		else {
			info = S.h.ltype | (S.nseq ? ZDS_I_SEQ : 0u) | (S.modes << 8);
			nseq = S.nseq;
			regen = S.h.regen;
		}
	}
	blk[g].info = info;
	blk[g].nseq = nseq;
	blk[g].lit_regen = regen;
}
// 3. table sources (thread per frame): Treeless literals use the Huffman tree of the last block that carried one;
//    Repeat_Mode uses the table of the last block with sequences, whatever its mode was (RFC 8878 3.1.1.3.2.1).
__global__ void __launch_bounds__(128)
k_zds_sources(const u32* __restrict__ multi, u64 nmulti, const u64* __restrict__ first, const u32* __restrict__ nblk, ZdsBlk* __restrict__ blk) {
	u64 m = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (m >= nmulti) return;
	u32 k = multi[m];
	u64 f0 = first[k];
	u32 nb = nblk[k];
	u32 last[4] = {ZDS_NONE, ZDS_NONE, ZDS_NONE, ZDS_NONE};
	for (u32 j = 0; j < nb; j++) {
		u64 g = f0 + j;
		u32 hdr = blk[g].hdr, info = blk[g].info;
		u32 src[4] = {ZDS_NONE, ZDS_NONE, ZDS_NONE, ZDS_NONE};
		if (((hdr >> 1) & 3) == 2 && !(info & ZDS_I_BAD)) {
			u32 lt = info & ZDS_I_LTYPE;
			if (lt == 2) last[0] = (u32)g;
			if (lt >= 2) src[0] = last[0];
			if (info & ZDS_I_SEQ) {
				u32 modes = ZDS_I_MODES(info);
				for (u32 t = 0; t < 3; t++) {  // LL (bits 7-6), OF (5-4), ML (3-2) -> slots 1, 2, 3
					u32 mode = (modes >> (6 - 2 * t)) & 3;
					if (mode != 3) last[1 + t] = (u32)g;
					src[1 + t] = last[1 + t];
				}
			}
		}
		for (u32 t = 0; t < 4; t++) blk[g].src[t] = src[t];
	}
}

// ---------------------------------------------------------------------------------------------
// chunk items: the blocks with index in [J, J + w) of every staged frame, ordered by block index (so that the
// executor's in-order hand-out serves all frames side by side).  jbase[j] = position of the first item with block
// index j inside its chunk (host-computed from the histogram of block counts); cursor[j] starts at 0.
__global__ void __launch_bounds__(128)
k_zds_chunk_items(const u32* __restrict__ multi, u64 nmulti, const u64* __restrict__ first, const u32* __restrict__ nblk,
                  const ZdsBlk* __restrict__ blk, u32 J, u32 w, const u32* __restrict__ jbase, u32* __restrict__ cursor, u32* __restrict__ items,
                  u32* __restrict__ item_of, u64* __restrict__ seq_cnt, u64* __restrict__ lit_cnt) {
	u64 m = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
	if (m >= nmulti) return;
	u32 k = multi[m];
	u32 nb = nblk[k];
	if (nb <= J) return;
	u64 f0 = first[k];
	u32 hi = zg_min<u32>(nb, J + w);
	for (u32 j = J + zg_lane(); j < hi; j += 32) {
		u32 pos = jbase[j] + atomicAdd(&cursor[j], 1u);
		u64 g = f0 + j;
		items[pos] = (u32)g;
		item_of[g] = pos;
		u32 info = blk[g].info;
		seq_cnt[pos] = blk[g].nseq;
		lit_cnt[pos] = ((info & ZDS_I_LTYPE) >= 2 && !(info & ZDS_I_BAD)) ? (u64)((blk[g].lit_regen + 15u) & ~15u) : 0ull;
	}
}

// ---------------------------------------------------------------------------------------------
// 4. entropy stage
// one of the three sequence tables of the block `self` (sections S): its own description when the mode says so, else
// the description in the block `from` (sections F) that last defined it.  Uniform in the warp.
ZG_DEV bool zds_table(ZdWarp* W, u32* slot, u32& log, u32& flags, u32 ok_flag, u32 def_flag, u32 t, u32 mode, const u8*& p, const u8* end,
                      const u8* fsrc, u32 fn, u32 maxlog, u32 maxsym, u32 def_log) {
	if (mode != 3) return zd_seq_table(W, slot, log, flags, ok_flag, def_flag, mode, p, end, maxlog, maxsym, def_log);
	if (!fsrc) return false;  // Repeat_Mode with nothing to repeat
	ZdsSect F;
	if (!zds_sections(fsrc, fn, F) || F.nseq == 0) return false;
	const u8* q = F.tables;
	const u8* qend = fsrc + fn;
	// skip the descriptions in front of table t (order LL, OF, ML)
	const u32 mlog[3] = {ZS_LL_MAXLOG, ZS_OF_MAXLOG, ZS_ML_MAXLOG}, msym[3] = {35, 31, 52};
	for (u32 u = 0; u < t; u++) {
		u32 um = (F.modes >> (6 - 2 * u)) & 3;
		if (um == 1) q += 1;
		else if (um == 2) {
			if (zg_lane() == 0) {
				u32 nsym = 0, lg = 0;
				W->misc[0] = q < qend ? zs_read_ncount(q, (u32)(qend - q), mlog[u], msym[u], W->norm, &nsym, &lg) : 0u;
			}
			__syncwarp();
			u32 nc = W->misc[0];
			__syncwarp();
			if (nc == 0) return false;
			q += nc;
		}
		if (q > qend) return false;
	}
	u32 fm = (F.modes >> (6 - 2 * t)) & 3;
	if (fm == 3) return false;  // (the source is, by construction, a block that defined the table)
	return zd_seq_table(W, slot, log, flags, ok_flag, def_flag, fm, q, qend, maxlog, maxsym, def_log);
}

// Huffman literals of one block into dst (uniform).  `tsrc`/`tn`: the block whose tree a Treeless block uses.
ZG_DEV_NOINLINE u32 zds_literals(ZdWarp* W, const u8* src, const ZdLitHdr& h, const u8* tsrc, u32 tn, u8* dst) {
	u32 lane = zg_lane();
	const u8* lp = src + h.hdr;
	const u8* lend = lp + h.comp;
	u32 nw = 0, huf_bits;
	if (h.ltype == 2) {
		u32 used = zd_read_huf_weights(W, lp, h.comp, &nw);
		if (used == 0) return ZS_E_CORRUPT;
		lp += used;
	} else {
		ZdLitHdr th;
		if (!tsrc || !zd_lit_header(tsrc, tn, th) || th.ltype != 2) return ZS_E_CORRUPT;
		if (zd_read_huf_weights(W, tsrc + th.hdr, th.comp, &nw) == 0) return ZS_E_CORRUPT;
	}
	huf_bits = zd_build_huf(W, nw);
	if (huf_bits == 0) return ZS_E_CORRUPT;
	u32 regen = h.regen;
	bool ok = true;
	if (h.streams == 1) {
		if (lane == 0) ok = zd_huf_stream(W->huf, huf_bits, lp, (u32)(lend - lp), dst, regen);
	} else {
		if (lend - lp < 10) return ZS_E_CORRUPT;
		u32 s1 = zg_ld16(lp), s2 = zg_ld16(lp + 2), s3 = zg_ld16(lp + 4);
		lp += 6;
		u32 avail = (u32)(lend - lp);
		u32 seg = (regen + 3) >> 2;
		if (s1 + s2 + s3 >= avail || seg * 3 > regen) return ZS_E_CORRUPT;
		if (lane < 4) {
			u32 so = lane == 0 ? 0 : lane == 1 ? s1 : lane == 2 ? s1 + s2 : s1 + s2 + s3;
			u32 sn = lane == 0 ? s1 : lane == 1 ? s2 : lane == 2 ? s3 : avail - s1 - s2 - s3;
			u32 cnt = lane < 3 ? seg : regen - 3 * seg;
			ok = zd_huf_stream(W->huf, huf_bits, lp + so, sn, dst + lane * seg, cnt);
		}
	}
	if (!__all_sync(ZG_FULL, ok)) return ZS_E_CORRUPT;
	__syncwarp();
	return ZS_OK;
}

// the lane-private state of one block in the entropy stage
struct ZdsLane {
	ZsBack b;
	u32 sl, so, sm;
	u32 ll_log, ml_log, of_log;
	u32 flags;          // ZD_F_*_DEF
	u32 nseq, left;
	u32 status;
	u32 rep0, rep1, rep2;
	u32 pos, lit_used;  // bytes regenerated / literals consumed by the sequences so far
	i32 reach;          // furthest a concrete offset went below the block's first byte
	u32 sym;            // a symbolic offset was used
};

// `cnt` sequences of this lane's block -> dst, packed like the fused decoder's (offset:28 | litLength:18 | matchLength:18);
// the loop body is zd_lane_decode's, with the offsets checked against the window and the block's reach tracked
ZG_DEV bool zds_lane_decode(ZdsLane& L, u32 cnt, const u32* llt, const u32* mlt, const u32* oft, u64* dst) {
	ZsBack b = L.b;
	u32 sl = L.sl, so = L.so, sm = L.sm;
	u32 rep0 = L.rep0, rep1 = L.rep1, rep2 = L.rep2;
	u32 left = L.left, pos = L.pos, lit_used = L.lit_used, sym = L.sym;
	i32 reach = L.reach;
	ZsBelow ahead = {0, 0};
	zs_below_fetch(b, ahead);
	u32 bad = 0;
	for (u32 k = 0; k < cnt; k++) {
		u32 oe = oft[so], me = mlt[sm], le = llt[sl];
		zs_back_reload_ahead(b, ahead);
		u32 oc = oe & 0xff;
		u32 mp = ZS_ML_PACK[me & 0xff], lp = ZS_LL_PACK[le & 0xff];
		u32 ofv = (1u << oc) + zs_back_read(b, oc);
		u32 used = oc;
		if (oc > 24) {
			zs_back_reload_ahead(b, ahead);
			used = 0;
		}
		u32 mb = mp >> 24, lb = lp >> 24;
		u32 ml = (mp & 0xffffffu) + zs_back_read(b, mb);
		u32 ll = (lp & 0xffffffu) + zs_back_read(b, lb);
		used += mb + lb;
		if (left - k > 1) {
			if (used > 30) zs_back_reload_ahead(b, ahead);
			sl = (le >> 16) + zs_back_read(b, (le >> 8) & 0xff);
			sm = (me >> 16) + zs_back_read(b, (me >> 8) & 0xff);
			so = (oe >> 16) + zs_back_read(b, (oe >> 8) & 0xff);
		}
		u32 off;
		if (ofv > 3) {
			off = ofv - 3;
			bad |= off > ZDS_WIN_MAX ? 1u : 0u;  // beyond every window this decoder accepts (and the symbolic range starts here)
			rep2 = rep1;
			rep1 = rep0;
			rep0 = off;
		} else {
			u32 idx = ofv - 1 + (ll == 0 ? 1 : 0);
			off = idx == 0 ? rep0 : idx == 1 ? rep1 : idx == 2 ? rep2 : rep0 - 1u;
			if (idx > 1) rep2 = rep1;
			if (idx > 0) {
				rep1 = rep0;
				rep0 = off;
			}
			// "rep0 - 1" of a concrete 1 is no offset; of a symbolic value it stays symbolic as long as the block has
			// fewer than 2^25 sequences (it has at most ZDS_MAXSEQ)
			bad |= off == 0u ? 1u : 0u;
		}
		pos += ll;
		lit_used += ll;
		bool s = zds_is_sym(off);
		sym |= s ? 1u : 0u;
		i32 r = (i32)off - (i32)pos;
		reach = (!s && r > reach) ? r : reach;
		pos += ml;
		dst[k] = (u64)off | ((u64)ll << 28) | ((u64)ml << 46);
	}
	if (bad || zs_back_overflow(b)) return false;
	left -= cnt;
	if (left == 0) {
		zs_back_reload(b);
		if (!zs_back_finished(b)) return false;
	}
	L.b = b;
	L.sl = sl;
	L.so = so;
	L.sm = sm;
	L.rep0 = rep0;
	L.rep1 = rep1;
	L.rep2 = rep2;
	L.left = left;
	L.pos = pos;
	L.lit_used = lit_used;
	L.reach = reach;
	L.sym = sym;
	return true;
}

struct ZdsJob {
	const u8* archive;
	const u64* off;       // per frame
	const u64* len;
	const u64* ulen;
	const u64* out_off;
	u8* out;
	const ZdsBlk* blk;
	ZdsRes* res;
	const u32* items;     // this chunk's blocks, by block index
	u32 nitems;
	const u64* seq_off;   // per item of the chunk: first sequence / first literal byte in the staging
	const u64* lit_off;
	u64* seq_stage;
	u8* lit_stage;
	// frame scan / execution
	u64* out_pos;         // per block: output offset inside its frame
	u32* rep_in;          // per block: the three repeat offsets it starts with
	u32* dep;             // per block: first block (index in frame) whose output it reads; == j: none
	u32* done;            // per block: executed
	u32* done_upto;       // per frame: all blocks below this index are executed (a hint that only grows)
	u32* f_status;        // per frame: first error
	u32* f_chain;         // per frame: a block of this chunk reads earlier blocks (the frame goes to the chain executor)
	u32* item_of;         // per block: its position among the chunk's items
};

__global__ void __launch_bounds__(ZDS_WARPS * 32, ZDS_ENT_CTAS)
k_zds_entropy(ZdsJob J, u32* tabs, u32* queue, u32 want) {
	ZG_DYN_SMEM(ZdWarp, sm);
	u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	ZdWarp* W = &sm[warp];
	size_t gw = (size_t)blockIdx.x * ZDS_WARPS + warp;
	u32* my_slot = tabs + (gw * 32 + lane) * ZD_TAB_SLOT;
	for (;;) {
		u32 base = 0;
		if (lane == 0) base = atomicAdd(queue, want);
		base = __shfl_sync(ZG_FULL, base, 0);
		if (base >= J.nitems) break;
		bool mine = lane < want && base + lane < J.nitems;
		u32 i = mine ? base + lane : 0;
		u32 g = mine ? J.items[i] : 0;
		ZdsBlk B;
		B.hdr = 0;
		B.info = 0;
		if (mine) B = J.blk[g];
		u32 type = (B.hdr >> 1) & 3, bsize = B.hdr >> 3;
		ZdsLane L;
		L.b.start = L.b.ptr = J.archive;
		L.b.lo = L.b.hi = L.b.consumed = 0;
		L.sl = L.so = L.sm = 0;
		L.ll_log = L.ml_log = L.of_log = 0;
		L.flags = 0;
		L.nseq = L.left = 0;
		L.status = ZS_OK;
		L.rep0 = zds_sym(0);
		L.rep1 = zds_sym(1);
		L.rep2 = zds_sym(2);
		L.pos = L.lit_used = 0;
		L.reach = 0;
		L.sym = 0;
		u32 regen = 0;
		if (mine && type != 2) regen = bsize;                       // Raw / RLE block
		if (mine && type == 2 && (B.info & ZDS_I_BAD)) L.status = ZS_E_CORRUPT;
		// ---- A: tables, bitstream start and literals of every compressed block, one block at a time ----
		u32 todo = __ballot_sync(ZG_FULL, mine && type == 2 && L.status == ZS_OK);
		while (todo) {
			int f = __ffs((int)todo) - 1;
			todo &= todo - 1;
			u32 gf = __shfl_sync(ZG_FULL, g, f), itf = __shfl_sync(ZG_FULL, i, f);
			ZdsBlk U = J.blk[gf];
			const u8* fsrc = J.archive + J.off[U.k];
			const u8* body = fsrc + U.ip + 3;
			u32 n = U.hdr >> 3;
			ZdsSect S;
			zds_sections(body, n, S);  // validated by k_zds_modes
			u32 st = ZS_OK;
			// literals (Raw and RLE literals are read in place by the executor)
			if (S.h.ltype >= 2) {
				const u8* tsrc = nullptr;
				u32 tn = 0;
				if (S.h.ltype == 3 && U.src[0] != ZDS_NONE) {
					ZdsBlk T = J.blk[U.src[0]];
					tsrc = fsrc + T.ip + 3;
					tn = T.hdr >> 3;
				}
				st = zds_literals(W, body, S.h, tsrc, tn, J.lit_stage + J.lit_off[itf]);
			}
			ZdsLane V = L;  // (uniform copy of the fields the set-up writes; lane f keeps it)
			V.nseq = V.left = S.nseq;
			if (st == ZS_OK && S.nseq) {
				const u8* p = S.tables;
				const u8* end = body + n;
				u32* slot = tabs + (gw * 32 + (u32)f) * ZD_TAB_SLOT;
				u32 fl = 0;
				bool ok = true;
				const u32 maxlog[3] = {ZS_LL_MAXLOG, ZS_OF_MAXLOG, ZS_ML_MAXLOG}, maxsym[3] = {35, 31, 52}, deflog[3] = {6, 5, 6};
				const u32 okf[3] = {ZD_F_LL_OK, ZD_F_OF_OK, ZD_F_ML_OK}, deff[3] = {ZD_F_LL_DEF, ZD_F_OF_DEF, ZD_F_ML_DEF};
				const u32 slotoff[3] = {0, 1024, 512};
				u32 logs[3] = {0, 0, 0};
				for (u32 t = 0; t < 3 && ok; t++) {
					u32 mode = (S.modes >> (6 - 2 * t)) & 3;
					const u8* ts = nullptr;
					u32 tn = 0;
					if (mode == 3 && U.src[1 + t] != ZDS_NONE) {
						ZdsBlk T = J.blk[U.src[1 + t]];
						ts = fsrc + T.ip + 3;
						tn = T.hdr >> 3;
					}
					ok = zds_table(W, slot + slotoff[t], logs[t], fl, okf[t], deff[t], t, mode, p, end, ts, tn, maxlog[t], maxsym[t], deflog[t]);
				}
				if (ok) {
					V.ll_log = logs[0];
					V.of_log = logs[1];
					V.ml_log = logs[2];
					V.flags = fl;
					ok = zs_back_init(V.b, p, (u32)(end - p));
					if (ok) {
						zs_back_reload(V.b);
						V.sl = zs_back_read(V.b, V.ll_log);
						V.so = zs_back_read(V.b, V.of_log);
						V.sm = zs_back_read(V.b, V.ml_log);
						ok = !zs_back_overflow(V.b);
					}
				}
				if (!ok) st = ZS_E_CORRUPT;
			}
			V.status = st;
			if (st != ZS_OK) V.nseq = V.left = 0;
			if (lane == (u32)f) L = V;
			__syncwarp();
		}
		// ---- B: every lane decodes its block's sequences (in bounded steps, so the warp reconverges) ----
		{
			const u32* llt = (L.flags & ZD_F_LL_DEF) ? ZS_LL_DEFAULT_DTABLE : my_slot;
			const u32* mlt = (L.flags & ZD_F_ML_DEF) ? ZS_ML_DEFAULT_DTABLE : my_slot + 512;
			const u32* oft = (L.flags & ZD_F_OF_DEF) ? ZS_OF_DEFAULT_DTABLE : my_slot + 1024;
			u64* dst = J.seq_stage + (mine ? J.seq_off[i] : 0);
			for (;;) {
				u32 cnt = zg_min<u32>(64u, L.left);
				if (!__any_sync(ZG_FULL, cnt > 0)) break;
				if (cnt && !zds_lane_decode(L, cnt, llt, mlt, oft, dst + (L.nseq - L.left))) {
					L.status = ZS_E_CORRUPT;
					L.left = 0;
				}
			}
		}
		__syncwarp();
		if (mine) {
			if (type == 2 && L.status == ZS_OK) {
				// all literals are emitted: those between the matches and the rest after the last sequence
				if (L.lit_used > B.lit_regen) L.status = ZS_E_CORRUPT;
				else {
					regen = L.pos + (B.lit_regen - L.lit_used);
					if (regen > ZS_BLOCK_MAX) L.status = ZS_E_CORRUPT;
				}
			}
			ZdsRes R;
			R.status = L.status;
			R.regen = L.status == ZS_OK ? regen : 0;
			R.rep[0] = L.rep0;
			R.rep[1] = L.rep1;
			R.rep[2] = L.rep2;
			R.need_back = L.reach > 0 ? (u32)L.reach : 0u;
			R.flags = L.sym ? ZDS_R_SYM : 0u;
			R.lit_used = L.lit_used;
			J.res[g] = R;
		}
		__syncwarp();
	}
}

// ---------------------------------------------------------------------------------------------
// 5. frame scan over the chunk's range of block indices (thread per frame): output offsets, incoming histories,
//    and which earlier block each block has to wait for.
__global__ void __launch_bounds__(128)
k_zds_frame_scan(ZdsJob J, const u32* __restrict__ multi, u64 nmulti, const u64* __restrict__ first, const u32* __restrict__ nblk, u32 J0, u32 w,
                 u64* __restrict__ f_out, u32* __restrict__ f_rep, u32* __restrict__ chain_list, unsigned long long* chain_count) {
	u64 m = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (m >= nmulti) return;
	u32 k = multi[m];
	u32 nb = nblk[k];
	if (nb <= J0) return;
	u64 f0 = first[k];
	u32 hi = zg_min<u32>(nb, J0 + w);
	u64 o = f_out[k], cap = J.ulen[k];
	u32 r0 = f_rep[3 * (u64)k], r1 = f_rep[3 * (u64)k + 1], r2 = f_rep[3 * (u64)k + 2];
	u32 st = J.f_status[k];
	bool chained = false;
	for (u32 j = J0; j < hi; j++) {
		u64 g = f0 + j;
		ZdsRes R = J.res[g];
		if (st == ZS_OK && R.status != ZS_OK) st = R.status;
		if (st == ZS_OK && o + R.regen > cap) st = ZS_E_DST_SMALL;
		J.out_pos[g] = o;
		J.rep_in[3 * g] = r0;
		J.rep_in[3 * g + 1] = r1;
		J.rep_in[3 * g + 2] = r2;
		// the first block whose output this one reads: everything when the reach is not known (offsets out of the
		// incoming history), else the block holding byte o - need_back (binary search over the offsets so far)
		u32 dj = j;
		if (R.flags & ZDS_R_SYM) dj = 0;
		else if (R.need_back) {
			u64 want = o > R.need_back ? o - R.need_back : 0;
			u32 lo = 0, hh = j;  // first block ending after `want`
			while (lo < hh) {
				u32 mid = (lo + hh) >> 1;
				u64 e = mid + 1 < j ? J.out_pos[f0 + mid + 1] : o;  // end of block mid = start of block mid + 1
				if (e > want) hh = mid;
				else lo = mid + 1;
			}
			dj = lo;
		}
		J.dep[g] = dj;
		chained = chained || dj < j;
		if (st == ZS_OK) {
			u32 n0 = zds_resolve(R.rep[0], r0, r1, r2), n1 = zds_resolve(R.rep[1], r0, r1, r2), n2 = zds_resolve(R.rep[2], r0, r1, r2);
			r0 = n0;
			r1 = n1;
			r2 = n2;
			o += R.regen;
		}
	}
	f_out[k] = o;
	f_rep[3 * (u64)k] = r0;
	f_rep[3 * (u64)k + 1] = r1;
	f_rep[3 * (u64)k + 2] = r2;
	J.f_status[k] = st;
	J.f_chain[k] = chained ? 1u : 0u;
	if (chained && st == ZS_OK) chain_list[atomicAdd(chain_count, 1ull)] = k;
}

// ---------------------------------------------------------------------------------------------
// 6. execution
// a word another warp may be writing: read once per warp (lane 0) so that all lanes act on the same value
ZG_DEV u32 zds_ld_flag(const u32* p) { return *(const volatile u32*)p; }
ZG_DEV u32 zds_ld_flag_warp(const u32* p) {
	u32 v = zg_lane() == 0 ? zds_ld_flag(p) : 0u;
	return __shfl_sync(ZG_FULL, v, 0);
}
ZG_DEV void zds_backoff() {
#ifdef ZG_EMU
	zg_emu::yield();
#else
	__nanosleep(64);
#endif
}
// wait until blocks [dj, j) of the frame (flags at done + f0) are executed.  The frame's done_upto only grows and
// always names a fully executed prefix, so the scan starts there.
ZG_DEV void zds_wait(const u32* done, u32* done_upto, u64 f0, u32 k, u32 dj, u32 j) {
	u32 lane = zg_lane();
	u32 p = zds_ld_flag_warp(&done_upto[k]);
	bool prefix = dj <= p;  // then what this warp verifies extends the known prefix
	p = zg_max<u32>(p, dj);
	while (p < j) {
		u32 q = p + lane;
		bool set = q >= j || zds_ld_flag(&done[f0 + q]) != 0;
		u32 miss = __ballot_sync(ZG_FULL, !set);
		if (miss == 0) p = zg_min<u32>(p + 32, j);
		else {
			p += (u32)__ffs((int)miss) - 1u;
			if (lane == 0) zds_backoff();
			__syncwarp();
		}
	}
	if (prefix && lane == 0) atomicMax(&done_upto[k], j);
	__threadfence();  // acquire: the copies below must see what the flagged blocks wrote
}

// Phase C of one block: zd_exec_row with the symbolic offsets made concrete first, and with L2 (CG) loads for the match
// sources, which other SMs may have written during this kernel.
__global__ void __launch_bounds__(ZDS_WARPS * 32, ZDS_EXEC_CTAS)
k_zds_exec(ZdsJob J, const u64* __restrict__ first, u32* queue, u32 skip_chained) {
	u32 lane = threadIdx.x & 31;
	for (;;) {
		u32 i = 0;
		if (lane == 0) i = atomicAdd(queue, 1u);
		i = __shfl_sync(ZG_FULL, i, 0);
		if (i >= J.nitems) break;
		u32 g = J.items[i];
		ZdsBlk B = J.blk[g];
		ZdsRes R = J.res[g];
		u32 k = B.k, j = B.j;
		u64 f0 = first[k];
		if (skip_chained && J.f_chain[k]) continue;  // the chain executor's (nothing in this chunk waits on its flags)
		u32 st = zds_ld_flag_warp(&J.f_status[k]);
		if (st == ZS_OK && R.status == ZS_OK) {
			u32 dj = J.dep[g];
			if (dj < j) zds_wait(J.done, J.done_upto, f0, k, dj, j);
			const u8* fsrc = J.archive + J.off[k];
			const u8* body = fsrc + B.ip + 3;
			u8* out = J.out + J.out_off[k];
			u64 o = J.out_pos[g], cap = J.ulen[k];
			u32 type = (B.hdr >> 1) & 3, bsize = B.hdr >> 3;
			u32 err = ZS_OK;
			if (type == 0) zg_warp_copy(out + o, body, bsize);
			else if (type == 1) zg_warp_fill(out + o, body[0], bsize);
			else {
				ZdLitHdr h;
				zd_lit_header(body, bsize, h);  // validated by k_zds_modes
				const u8* lit = h.ltype == 0 ? body + h.hdr : h.ltype == 1 ? body : J.lit_stage + J.lit_off[i];
				bool lit_rle = h.ltype == 1;
				u32 rle_byte = lit_rle ? body[h.hdr] : 0;
				u32 r0 = J.rep_in[3 * (u64)g], r1 = J.rep_in[3 * (u64)g + 1], r2 = J.rep_in[3 * (u64)g + 2];
				const u64* seqs = J.seq_stage + J.seq_off[i];
				u32 lpos = 0;
				u32 nseq = B.nseq;
				u64 sq = lane < nseq ? seqs[lane] : 0;
				for (u32 s0 = 0; s0 < nseq && err == ZS_OK; s0 += 32) {
					u64 sq_next = s0 + 32 + lane < nseq ? seqs[s0 + 32 + lane] : 0;
					// offsets out of the incoming history become concrete here
					u32 of = (u32)sq & ZD_OFF_MAX;
					bool act = s0 + lane < nseq;
					u32 rof = zds_resolve(of, r0, r1, r2);
					if (__any_sync(ZG_FULL, act && rof == 0)) err = ZS_E_CORRUPT;
					else {
						sq = (sq & ~(u64)ZD_OFF_MAX) | rof;
						err = zd_exec_row(sq, zg_min<u32>(32u, nseq - s0), ZdDirect<true>{out}, o, 0, cap, lit, lit_rle, rle_byte, h.regen, lpos);
					}
					sq = sq_next;
				}
				if (err == ZS_OK) {
					u32 rest = h.regen - lpos;
					if (o + rest > cap) err = ZS_E_DST_SMALL;
					else if (rest) {
						if (lit_rle) zg_warp_fill(out + o, rle_byte, rest);
						else zg_warp_copy(out + o, lit + lpos, rest);
					}
				}
			}
			if (err != ZS_OK && lane == 0) atomicCAS(&J.f_status[k], (u32)ZS_OK, err);
		}
		__syncwarp();
		__threadfence();  // release: this block's bytes before its flag
		if (lane == 0) *(volatile u32*)&J.done[g] = 1u;
	}
}


// ---------------------------------------------------------------------------------------------
// 6b. the chain executor.  A frame whose blocks read earlier blocks is a chain: every match may need bytes the matches just
// before it produced, and through global memory each such hop costs an L2 round trip (~700 cycles store-to-load; measured
// 100 MB/s per frame).  Here ONE warp walks the frame's blocks in order and keeps the recent output in a SHARED-MEMORY
// WINDOW: sequence execution happens in shared memory (a hop is a shared-memory round trip), the window is written to the
// frame's place in global memory with coalesced 16-byte stores when it slides, and only matches that reach back beyond the
// window read global memory (old bytes, off the critical path).
#define ZDC_CAP (64u << 10)    // window bytes
#define ZDC_HIST (16u << 10)   // history kept when the window slides
struct ZdWindow {
	uintptr_t bias;  // shared-memory address frame position q maps to is bias + q, for q in [lo, written)
	u64 lo;          // positions below are in global memory only (and everything below `lo` IS there)
	const u8* g;     // the frame's output in global memory
	ZG_DEV u8* dst(u64 pos) const { return (u8*)(bias + (uintptr_t)pos); }
	ZG_DEV void lane_copy(u64 dpos, u64 spos, u32 n) const {
		for (u32 k0 = 0; k0 < n; k0 += 16) {
			u64 q = spos + k0;
			u32 m = zg_min<u32>(16u, n - k0);
			u8* dp = dst(dpos + k0);
			if (q >= lo) zd_lane_copy<false>(dp, (const u8*)dst(q), m);
			else if (q + m <= lo) zd_lane_copy<true>(dp, g + q, m);
			else
				for (u32 i = 0; i < m; i++) dp[i] = q + i >= lo ? *dst(q + i) : (u8)zd_ldb<true>(g + q + i);
		}
	}
	ZG_DEV void lane_overlap(u64 dpos, u32 off, u32 ml) const {
		u32 done = 0;
		while (done < ml) {
			u32 c = zg_min<u32>(done + off, ml - done);
			lane_copy(dpos + done, dpos - off, c);
			done += c;
		}
	}
	ZG_DEV void warp_copy(u64 dpos, u64 spos, u32 n) const {
		u32 far = spos < lo ? (u32)zg_min<u64>(n, lo - spos) : 0u;
		if (far) zg_warp_copy_t<true>(dst(dpos), g + spos, far);
		if (n > far) zg_warp_copy_t<false>(dst(dpos + far), (const u8*)dst(spos + far), n - far);
	}
	ZG_DEV void warp_match(u64 dpos, u32 off, u32 ml) const {  // off < ml: the first period, then the match feeds on itself
		warp_copy(dpos, dpos - off, off);
		__syncwarp();
		zd_warp_match<false>(dst(dpos + off), off, ml - off);
	}
};

struct ZdcState {
	u8* buf;        // the window's shared memory (ZDC_CAP + 32 bytes, 16-byte aligned)
	u8* gout;       // the frame's output in global memory
	u64 abase;      // frame position of buf[0] (a multiple of 16)
	u64 lo;         // see ZdWindow
	u64 flushed;    // positions below are in global memory
};
ZG_DEV ZdWindow zdc_window(const ZdcState& S) { return ZdWindow{(uintptr_t)S.buf - (uintptr_t)S.abase, S.lo, S.gout}; }
// everything produced so far into global memory
ZG_DEV void zdc_flush(ZdcState& S, u64 pos) {
	if (pos > S.flushed) zg_warp_copy(S.gout + S.flushed, S.buf + (S.flushed - S.abase), (u32)(pos - S.flushed));
	S.flushed = pos;
	__syncwarp();
}
// make room for `need` more bytes at `pos`: false when they cannot fit the window at all (the caller then works in global memory)
ZG_DEV bool zdc_room(ZdcState& S, u64 pos, u32 need) {
	if (pos + need <= S.abase + ZDC_CAP) return true;
	if (need > ZDC_CAP - ZDC_HIST - 16u) return false;
	zdc_flush(S, pos);
	// slide: keep the last ZDC_HIST bytes (what the matches right ahead are most likely to read)
	u64 nlo = zg_max<u64>(S.lo, pos > ZDC_HIST ? pos - ZDC_HIST : 0);
	u64 nab = nlo & ~(u64)15;
	u32 keep = (u32)(pos - nab), shift = (u32)(nab - S.abase);
	u32 lane = zg_lane();
	if (shift) {
		for (u32 v0 = 0; v0 < keep; v0 += 512) {  // forward, 16 bytes per lane: reads of a round finish before its writes
			u32 v = v0 + 16 * lane;
			uint4 x = make_uint4(0, 0, 0, 0);
			if (v < keep) x = *(const uint4*)(S.buf + shift + v);
			__syncwarp();
			if (v < keep) *(uint4*)(S.buf + v) = x;
			__syncwarp();
		}
	}
	S.abase = nab;
	S.lo = nlo;
	return true;
}
// leave the window: what follows is written to global memory directly
ZG_DEV void zdc_reset(ZdcState& S, u64 pos_before, u64 pos_after) {
	zdc_flush(S, pos_before);
	S.abase = pos_after & ~(u64)15;
	S.lo = S.flushed = pos_after;
}

#ifdef ZG_EMU
__global__ void
#else
__global__ void __maxnreg__(128)
#endif
k_zds_chain(ZdsJob J, const u32* __restrict__ chain_list, u32 nchain, const u64* __restrict__ first, const u32* __restrict__ nblk, u32 J0, u32 w,
            u32* queue) {
	ZG_DYN_SMEM(u8, smem);
	u32 lane = threadIdx.x & 31;
	for (;;) {
		u32 ci = 0;
		if (lane == 0) ci = atomicAdd(queue, 1u);
		ci = __shfl_sync(ZG_FULL, ci, 0);
		if (ci >= nchain) break;
		u32 k = chain_list[ci];
		u64 f0 = first[k];
		u32 hi = zg_min<u32>(nblk[k], J0 + w);
		const u8* fsrc = J.archive + J.off[k];
		u64 cap = J.ulen[k];
		ZdcState S;
		S.buf = smem;
		S.gout = J.out + J.out_off[k];
		u64 pos = J.out_pos[f0 + J0];
		S.abase = pos & ~(u64)15;
		S.lo = S.flushed = pos;
		u32 err = zds_ld_flag_warp(&J.f_status[k]);
		for (u32 j = J0; j < hi && err == ZS_OK; j++) {
			u64 g = f0 + j;
			ZdsBlk B = J.blk[g];
			u32 type = (B.hdr >> 1) & 3, bsize = B.hdr >> 3;
			const u8* body = fsrc + B.ip + 3;
			u64 o = J.out_pos[g];
			if (type != 2) {
				// Raw / RLE block: straight to global memory, the window starts over behind it
				zdc_reset(S, o, o + bsize);
				if (type == 0) zg_warp_copy(S.gout + o, body, bsize);
				else zg_warp_fill(S.gout + o, body[0], bsize);
				__syncwarp();
				continue;
			}
			ZdLitHdr h;
			zd_lit_header(body, bsize, h);  // validated by k_zds_modes
			// this block's position among the chunk's items: its staging offsets are indexed by item
			u32 it = J.item_of[g];
			const u8* lit = h.ltype == 0 ? body + h.hdr : h.ltype == 1 ? body : J.lit_stage + J.lit_off[it];
			bool lit_rle = h.ltype == 1;
			u32 rle_byte = lit_rle ? body[h.hdr] : 0;
			u32 r0 = J.rep_in[3 * g], r1 = J.rep_in[3 * g + 1], r2 = J.rep_in[3 * g + 2];
			const u64* seqs = J.seq_stage + J.seq_off[it];
			u32 nseq = B.nseq, lpos = 0;
			u64 sq = lane < nseq ? seqs[lane] : 0;
			for (u32 s0 = 0; s0 < nseq && err == ZS_OK; s0 += 32) {
				u64 sq_next = s0 + 32 + lane < nseq ? seqs[s0 + 32 + lane] : 0;
				bool act = s0 + lane < nseq;
				u32 rof = zds_resolve((u32)sq & ZD_OFF_MAX, r0, r1, r2);
				u32 ll = (u32)(sq >> 28) & 0x3ffffu, ml = (u32)(sq >> 46);
				u32 row = zg_warp_sum(act ? ll + ml : 0u);
				if (__any_sync(ZG_FULL, act && rof == 0)) err = ZS_E_CORRUPT;
				else {
					sq = (sq & ~(u64)ZD_OFF_MAX) | rof;
					u32 cnt = zg_min<u32>(32u, nseq - s0);
					if (zdc_room(S, o, row)) err = zd_exec_row(sq, cnt, zdc_window(S), o, 0, cap, lit, lit_rle, rle_byte, h.regen, lpos);
					else {  // a row larger than the window: in global memory (matches of tens of KiB: the hop latency does not matter)
						u64 o0 = o;
						zdc_flush(S, o0);
						err = zd_exec_row(sq, cnt, ZdDirect<true>{S.gout}, o, 0, cap, lit, lit_rle, rle_byte, h.regen, lpos);
						__syncwarp();
						S.abase = o & ~(u64)15;
						S.lo = S.flushed = o;
					}
				}
				sq = sq_next;
			}
			if (err == ZS_OK) {
				u32 rest = h.regen - lpos;
				if (o + rest > cap) err = ZS_E_DST_SMALL;
				else if (rest) {
					if (zdc_room(S, o, rest)) {
						u8* d = zdc_window(S).dst(o);
						if (lit_rle) zg_warp_fill(d, rle_byte, rest);
						else zg_warp_copy(d, lit + lpos, rest);
					} else {
						zdc_reset(S, o, o + rest);
						if (lit_rle) zg_warp_fill(S.gout + o, rle_byte, rest);
						else zg_warp_copy(S.gout + o, lit + lpos, rest);
					}
					o += rest;
				}
			}
			__syncwarp();
			if (err == ZS_OK) pos = o;
		}
		if (err == ZS_OK) zdc_flush(S, pos);
		else if (lane == 0) atomicCAS(&J.f_status[k], (u32)ZS_OK, err);
		__syncwarp();
	}
}

// The Content_Checksum of the staged frames, piece by piece: after a chunk of blocks has been executed, the whole KiB
// chunks of every frame's output up to the watermark `wm` (a snapshot of f_out taken behind that chunk's execution) are
// absorbed into the frame's accumulators.  Runs on a side stream while the next chunk of blocks is decoded: XXH64 is a
// serial chain per frame (2 GB/s), so for a few huge frames it is as long as everything else together.
__global__ void __launch_bounds__(128)
k_zds_xxh64_partial(const u8* __restrict__ archive, const u64* __restrict__ off, const u8* __restrict__ out, const u64* __restrict__ out_off,
                    const u32* __restrict__ multi, u64 nmulti, const u64* __restrict__ wm, u64* __restrict__ xx_done, u64* __restrict__ xx_acc) {
	__shared__ u64 sb[4][XX_SB_WORDS];
	u64 m = (u64)blockIdx.x * 4 + (threadIdx.x >> 5);
	if (m >= nmulti) return;
	u32 lane = threadIdx.x & 31;
	u32 k = multi[m];
	if (!((archive[off[k] + 4] >> 2) & 1)) return;  // no Content_Checksum in this frame
	u64 c0 = xx_done[k], c1 = wm[k] >> XX_CHUNK_SHIFT;
	if (c1 <= c0) return;
	u64 acc = xx_warp_acc0();
	if (c0 && lane < 4) acc = xx_acc[4 * (u64)k + lane];
	acc = xx_warp_chunks(out + out_off[k], c0, c1, acc, sb[threadIdx.x >> 5]);
	if (lane < 4) xx_acc[4 * (u64)k + lane] = acc;
	if (lane == 0) xx_done[k] = c1;
}

// frame results, as the serial decoder reports them
__global__ void __launch_bounds__(128)
k_zds_finish(const u8* __restrict__ archive, const u64* __restrict__ off, const u64* __restrict__ len, const u64* __restrict__ ulen,
             const u32* __restrict__ multi, u64 nmulti, const u64* __restrict__ tail, const u64* __restrict__ f_out, const u32* __restrict__ f_status,
             u32* __restrict__ status, u64* __restrict__ produced, u32* __restrict__ cksums) {
	u64 m = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (m >= nmulti) return;
	u32 k = multi[m];
	const u8* src = archive + off[k];
	u32 st = f_status[k];
	u64 t = tail[k];
	bool has_ck = (src[4] >> 2) & 1;
	bool has_fcs = (src[4] >> 5) != 0;  // Frame_Content_Size_Flag or Single_Segment_Flag
	if (st == ZS_OK && has_ck && t + 4 > len[k]) st = ZS_E_SRC_SIZE;
	// (Frame_Content_Size, when present, equals ulen for every staged frame: a different total is the corruption the
	// serial decoder reports at the end of the frame.  Without it ulen is only the room there is -- zg_decompress passes
	// 128 KiB per block -- and the frame may end short of it, as it may on the serial path.)
	if (st == ZS_OK && has_fcs && f_out[k] != ulen[k]) st = ZS_E_CORRUPT;
	status[k] = st;
	produced[k] = st == ZS_OK ? f_out[k] : 0;
	cksums[2 * (u64)k] = (st == ZS_OK && has_ck) ? zg_ld32(src + t) : 0u;
	cksums[2 * (u64)k + 1] = (st == ZS_OK && has_ck) ? 1u : 0u;
}

// ---------------------------------------------------------------------------------------------
// frames of this many bytes and more are staged (two blocks at least)
static u64 g_zds_split_min = (u64)ZS_BLOCK_MAX + 1;
extern "C" void zg_internal_set_decode_split_min(u64 v) { g_zds_split_min = v ? v : (u64)ZS_BLOCK_MAX + 1; }
// 0: dependent blocks wait on per-block flags (k_zds_exec); 1: frames with dependent blocks go to the chain executor when
// they fit the machine; 2: always
static u32 g_zds_chain_mode = 1;
extern "C" void zg_internal_set_decode_chain_mode(u32 v) { g_zds_chain_mode = v; }
static u32 g_zds_chunk_items = ZDS_CHUNK_ITEMS;
extern "C" void zg_internal_set_decode_chunk_blocks(u32 v) { g_zds_chunk_items = v ? v : ZDS_CHUNK_ITEMS; }  // (tests shrink it)
// what the last zg_zstd_decode_run did: {frames, work items (frames + blocks of staged frames), frames decoded twice
// (always 0: there is no second pass any more), staged frames, staged blocks, blocks that read earlier blocks, chunks,
// frame-chunks run by the chain executor}
u64 g_zd_stats[8];
extern "C" void zg_internal_decode_stats(u64 out[3]) {
	for (int i = 0; i < 3; i++) out[i] = g_zd_stats[i];
}
extern "C" void zg_internal_decode_stats_ex(u64 out[8]) {
	for (int i = 0; i < 8; i++) out[i] = g_zd_stats[i];
}

__global__ void __launch_bounds__(256) k_zds_count_deps(const ZdsBlk* __restrict__ blk, const u32* __restrict__ dep, const u32* __restrict__ items, u32 n,
                                                         unsigned long long* out) {
	u32 i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	u32 g = items[i];
	if (dep[g] < blk[g].j) atomicAdd(out, 1ull);
}

size_t zd_fused_launch(cudaStream_t s, ZgZdWork& w, const u8* archive, u64 archive_len, const u64* off, const u64* len, const u64* ulen,
                       const u64* out_off, const u32* list, u64 count, u8* out, u64 out_cap, u32* status, u64* produced, u32* cksums);

size_t zg_zstd_decode_run(cudaStream_t s, ZgZdWork& w, const u8* archive, u64 archive_len, const u64* off, const u64* len,
                          const u64* ulen, const u64* out_off, u64 n, u8* out, u64 out_cap, u32* status, u64* produced,
                          u32* cksums, int verify_checksums) {
	if (n == 0) return 0;
	if (n >= 0xffffffffull) return ZG_ERR(ZG_error_GENERIC);
	for (int i = 0; i < 8; i++) g_zd_stats[i] = 0;
	g_zd_stats[0] = g_zd_stats[1] = n;
	ZgZdStaged& S = w.st;
	S.xx_n = 0;
	if (S.nblk.reserve(n * 4) || S.first.reserve(n * 8) || S.multi.reserve(n * 4) || S.single.reserve(n * 4) || S.tot.reserve(64) ||
	    S.hist.reserve(((size_t)ZDS_HMAX + 2) * 4) || w.h.reserve(64))
		return ZG_ERR(ZG_error_memory_allocation);
	cudaMemsetAsync(S.tot.p, 0, 64, s);
	cudaMemsetAsync(S.hist.p, 0, ((size_t)ZDS_HMAX + 2) * 4, s);
	u32 gn = (u32)((n + 127) / 128);
	unsigned long long* tot = (unsigned long long*)S.tot.p;
	ZG_LAUNCH(k_zds_count, gn, 128, 0, s, archive, archive_len, off, len, ulen, out_off, out_cap, n, g_zds_split_min, S.nblk.as<u32>(),
	          S.first.as<u64>(), S.multi.as<u32>(), S.single.as<u32>(), tot, S.hist.as<u32>());
	ZG_COUNT_LAUNCH();
	u64* h = w.h.as<u64>();
	if (zg_publish(s, S.tot.p, h, 32) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) return ZG_ERR(ZG_error_device);
	u64 nmulti = h[0], nblocks = h[1], max_nb = h[2], nsingle = h[3];
	if (nmulti == 0)  // no multi-block frame: the items are the frames
		return zd_fused_launch(s, w, archive, archive_len, off, len, ulen, out_off, nullptr, n, out, out_cap, status, produced, cksums);
	if (nblocks >= 0xffffffffull) return ZG_ERR(ZG_error_GENERIC);
	g_zd_stats[1] = nsingle + nblocks;
	g_zd_stats[3] = nmulti;
	g_zd_stats[4] = nblocks;
	// single-block frames (and whatever the walk refused: the serial decoder names the error) in the fused kernel
	if (nsingle) {
		size_t r = zd_fused_launch(s, w, archive, archive_len, off, len, ulen, out_off, S.single.as<u32>(), nsingle, out, out_cap, status,
		                           produced, cksums);
		if (zg_is_error(r)) return r;
	}
	// ---- staged frames ----
	if (S.blk.reserve(nblocks * sizeof(ZdsBlk)) || S.res.reserve(nblocks * sizeof(ZdsRes)) || S.out_pos.reserve(nblocks * 8) ||
	    S.rep_in.reserve(nblocks * 12) || S.dep.reserve(nblocks * 4) || S.done.reserve(nblocks * 4) || S.tail.reserve(n * 8) ||
	    S.f_out.reserve(n * 8) || S.f_rep.reserve(n * 12) || S.f_status.reserve(n * 4) || S.done_upto.reserve(n * 4) ||
	    S.jbase.reserve((max_nb + 1) * 4) || S.cursor.reserve((max_nb + 1) * 4) || S.hh.reserve((max_nb + 2) * 8) || S.queue.reserve(64) ||
	    S.f_chain.reserve(n * 4) || S.item_of.reserve(nblocks * 4) || S.chain_list.reserve(nmulti * 4))
		return ZG_ERR(ZG_error_memory_allocation);
	u32 gm = (u32)((nmulti + 127) / 128);
	ZG_LAUNCH(k_zds_emit, gm, 128, 0, s, archive, archive_len, off, len, ulen, out_off, out_cap, S.multi.as<u32>(), nmulti, g_zds_split_min,
	          S.first.as<u64>(), S.blk.as<ZdsBlk>(), S.tail.as<u64>(), S.f_out.as<u64>(), S.f_rep.as<u32>(), S.f_status.as<u32>(),
	          S.done_upto.as<u32>());
	ZG_LAUNCH(k_zds_modes, (u32)((nblocks + 127) / 128), 128, 0, s, archive, off, S.blk.as<ZdsBlk>(), nblocks);
	ZG_LAUNCH(k_zds_sources, gm, 128, 0, s, S.multi.as<u32>(), nmulti, S.first.as<u64>(), S.nblk.as<u32>(), S.blk.as<ZdsBlk>());
	g_zg_launches += 3;
	cudaMemsetAsync(S.done.p, 0, nblocks * 4, s);
	cudaMemsetAsync(S.cursor.p, 0, (max_nb + 1) * 4, s);
	// chunks: ranges [J, J + w) of block indices holding <= chunk_items blocks; cnt_ge[j] = frames with more than j blocks
	u32* hist = S.hh.as<u32>();                  // [max_nb + 1]
	u32* jb = hist + (max_nb + 2);               // [max_nb + 1] -> jbase
	if (cudaMemcpyAsync(hist, S.hist.p, (max_nb + 1) * 4, cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess)
		return ZG_ERR(ZG_error_device);
	struct Chunk {
		u32 J, w, items;
	};
	std::vector<Chunk> chunks;
	{
		std::vector<u32> cnt_ge(max_nb + 1, 0);
		u32 run = 0;
		for (u64 j = max_nb; j-- > 0;) {  // frames with nb > j
			run += hist[j + 1];
			cnt_ge[j] = run;
		}
		u64 Jc = 0;
		while (Jc < max_nb) {
			u32 wv = 0, it = 0;
			while (Jc + wv < max_nb && wv < ZDS_CHUNK_WIDTH && (wv == 0 || it + cnt_ge[Jc + wv] <= g_zds_chunk_items)) {
				jb[Jc + wv] = it;
				it += cnt_ge[Jc + wv];
				wv++;
			}
			chunks.push_back(Chunk{(u32)Jc, wv, it});
			Jc += wv;
		}
	}
	if (cudaMemcpyAsync(S.jbase.p, jb, max_nb * 4, cudaMemcpyHostToDevice, s) != cudaSuccess) return ZG_ERR(ZG_error_device);
	g_zd_stats[6] = chunks.size();
	u32 max_items = 0;
	for (auto& c : chunks) max_items = zg_max<u32>(max_items, c.items);
	if (S.items.reserve((size_t)max_items * 4) || S.seq_cnt.reserve((size_t)max_items * 8) || S.lit_cnt.reserve((size_t)max_items * 8) ||
	    S.seq_off.reserve((size_t)max_items * 8) || S.lit_off.reserve((size_t)max_items * 8))
		return ZG_ERR(ZG_error_memory_allocation);
	u32 sms = (u32)zg_sm_count();
	size_t smem = sizeof(ZdWarp) * ZDS_WARPS;
	static ZgPerDevice attr_dev;
	bool& attr_set = *attr_dev.slot();
	if (!attr_set) {
		if (cudaFuncSetAttribute(k_zds_entropy, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return ZG_ERR(ZG_error_device);
		attr_set = true;
	}
	ZdsJob J;
	J.archive = archive;
	J.off = off;
	J.len = len;
	J.ulen = ulen;
	J.out_off = out_off;
	J.out = out;
	J.blk = S.blk.as<ZdsBlk>();
	J.res = S.res.as<ZdsRes>();
	J.items = S.items.as<u32>();
	J.seq_off = S.seq_off.as<u64>();
	J.lit_off = S.lit_off.as<u64>();
	J.out_pos = S.out_pos.as<u64>();
	J.rep_in = S.rep_in.as<u32>();
	J.dep = S.dep.as<u32>();
	J.done = S.done.as<u32>();
	J.done_upto = S.done_upto.as<u32>();
	J.f_status = S.f_status.as<u32>();
	J.f_chain = S.f_chain.as<u32>();
	J.item_of = S.item_of.as<u32>();
	size_t smem_c = ZDC_CAP + 48;
	static ZgPerDevice attr_dev_c;
	bool& attr_set_c = *attr_dev_c.slot();
	if (!attr_set_c) {
		if (cudaFuncSetAttribute(k_zds_chain, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_c) != cudaSuccess) return ZG_ERR(ZG_error_device);
		attr_set_c = true;
	}
	u64* totals = (u64*)S.tot.p + 4;  // [4] sequences, [5] literal bytes, [6] blocks that wait
	cudaMemsetAsync(totals + 2, 0, 8, s);
	// Content_Checksums of the staged frames: hashed chunk by chunk on a side stream (k_zds_xxh64_partial), worth it when
	// the frames are few and long (several chunks); the check itself is zg_unpack_finalize_run's
	bool xx_side = false;
	if (verify_checksums && chunks.size() > 1) {
		if (!S.xx_init) {
			S.xx_init = true;
			if (cudaStreamCreateWithFlags(&S.xx_stream, cudaStreamNonBlocking) != cudaSuccess ||
			    cudaEventCreateWithFlags(&S.xx_fork, cudaEventDisableTiming) != cudaSuccess ||
			    cudaEventCreateWithFlags(&S.xx_join, cudaEventDisableTiming) != cudaSuccess)
				S.xx_fork = S.xx_join = nullptr;
		}
		if (S.xx_fork && S.xx_join && !S.xx_done.reserve(n * 8) && !S.xx_acc.reserve(n * 32) && !S.xx_wm.reserve(n * 8)) {
			xx_side = true;
			cudaMemsetAsync(S.xx_done.p, 0, n * 8, s);
		}
	}
	bool xx_pending = false;
	for (auto& c : chunks) {
		ZG_LAUNCH(k_zds_chunk_items, (u32)((nmulti + 3) / 4), 128, 0, s, S.multi.as<u32>(), nmulti, S.first.as<u64>(), S.nblk.as<u32>(),
		          S.blk.as<ZdsBlk>(), c.J, c.w, S.jbase.as<u32>(), S.cursor.as<u32>(), S.items.as<u32>(), S.item_of.as<u32>(), S.seq_cnt.as<u64>(),
		          S.lit_cnt.as<u64>());
		ZG_COUNT_LAUNCH();
		size_t r = zg_scan_run(s, w.tiles, S.seq_cnt.as<u64>(), c.items, 0, S.seq_off.as<u64>(), totals);
		if (!zg_is_error(r)) r = zg_scan_run(s, w.tiles, S.lit_cnt.as<u64>(), c.items, 0, S.lit_off.as<u64>(), totals + 1);
		if (zg_is_error(r)) return r;
		if (zg_publish(s, totals, h + 4, 16) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) return ZG_ERR(ZG_error_device);
		u64 nseq = h[4], nlit = h[5];
		if (S.seq_stage.reserve(nseq * 8 + 64) || S.lit_stage.reserve(nlit + 64)) return ZG_ERR(ZG_error_memory_allocation);
		J.nitems = c.items;
		J.seq_stage = S.seq_stage.as<u64>();
		J.lit_stage = S.lit_stage.as<u8>();
		// entropy: batches small enough that every warp gets a few
		u32 grid_e = (u32)zg_min<u64>(((u64)c.items + ZDS_WARPS - 1) / ZDS_WARPS, (u64)sms * ZDS_ENT_CTAS);
		u32 want = (u32)zg_min<u64>(32, zg_max<u64>(1, (u64)c.items / ((u64)grid_e * ZDS_WARPS * 3)));
		if (S.tabs.reserve((size_t)grid_e * ZDS_WARPS * 32 * ZD_TAB_SLOT * 4)) return ZG_ERR(ZG_error_memory_allocation);
		cudaMemsetAsync(S.queue.p, 0, 16, s);
		zg_prof_begin(ZG_K_DECODE, s);
		ZG_LAUNCH(k_zds_entropy, grid_e, ZDS_WARPS * 32, smem, s, J, S.tabs.as<u32>(), S.queue.as<u32>(), want);
		cudaMemsetAsync(totals + 3, 0, 8, s);
		ZG_LAUNCH(k_zds_frame_scan, gm, 128, 0, s, J, S.multi.as<u32>(), nmulti, S.first.as<u64>(), S.nblk.as<u32>(), c.J, c.w, S.f_out.as<u64>(),
		          S.f_rep.as<u32>(), S.chain_list.as<u32>(), (unsigned long long*)(totals + 3));
		// frames with blocks that read earlier blocks: by the chain executor (one warp and a shared-memory window per
		// frame) when they all fit the machine at once, else block by block behind per-block flags
		u64 nchain = 0;
		if (g_zds_chain_mode) {
			if (zg_publish(s, totals + 3, h + 7, 8) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) return ZG_ERR(ZG_error_device);
			nchain = h[7];
		}
		const u32 chain_slots = sms * (u32)(227u * 1024u / (ZDC_CAP + 1024u));
		bool use_chain = g_zds_chain_mode == 2 ? nchain > 0 : (nchain > 0 && nchain <= (u64)chain_slots * 4);
		g_zd_stats[7] += use_chain ? nchain : 0;
		u32 grid_x = (u32)zg_min<u64>(((u64)c.items + ZDS_WARPS - 1) / ZDS_WARPS, (u64)sms * ZDS_EXEC_CTAS);
		ZG_LAUNCH(k_zds_exec, grid_x, ZDS_WARPS * 32, 0, s, J, S.first.as<u64>(), S.queue.as<u32>() + 1, use_chain ? 1u : 0u);
		if (use_chain) {
			u32 grid_c = (u32)zg_min<u64>(nchain, (u64)chain_slots);
			ZG_LAUNCH(k_zds_chain, grid_c, 32, smem_c, s, J, S.chain_list.as<u32>(), (u32)nchain, S.first.as<u64>(), S.nblk.as<u32>(), c.J, c.w,
			          S.queue.as<u32>() + 2);
			ZG_COUNT_LAUNCH();
		}
		zg_prof_end(ZG_K_DECODE, s);
		if (xx_side) {
			// what this chunk produced can be hashed while the next chunk decodes: the watermarks are snapshot behind the
			// execution (f_out moves on with the next chunk's scan), once the side stream has finished with the last snapshot
			cudaStream_t sx = S.xx_stream ? S.xx_stream : s;
			if (xx_pending && cudaStreamWaitEvent(s, S.xx_join, 0) != cudaSuccess) return ZG_ERR(ZG_error_device);
			cudaMemcpyAsync(S.xx_wm.p, S.f_out.p, n * 8, cudaMemcpyDeviceToDevice, s);
			if (cudaEventRecord(S.xx_fork, s) != cudaSuccess || cudaStreamWaitEvent(sx, S.xx_fork, 0) != cudaSuccess) return ZG_ERR(ZG_error_device);
			ZG_LAUNCH(k_zds_xxh64_partial, (u32)((nmulti + 3) / 4), 128, 0, sx, archive, off, out, out_off, S.multi.as<u32>(), nmulti,
			          S.xx_wm.as<u64>(), S.xx_done.as<u64>(), S.xx_acc.as<u64>());
			ZG_COUNT_LAUNCH();
			if (cudaEventRecord(S.xx_join, sx) != cudaSuccess) return ZG_ERR(ZG_error_device);
			xx_pending = true;
		}
		ZG_LAUNCH(k_zds_count_deps, (c.items + 255) / 256, 256, 0, s, S.blk.as<ZdsBlk>(), S.dep.as<u32>(), S.items.as<u32>(), c.items,
		          (unsigned long long*)(totals + 2));
		g_zg_launches += 4;
	}
	if (xx_pending) {
		if (cudaStreamWaitEvent(s, S.xx_join, 0) != cudaSuccess) return ZG_ERR(ZG_error_device);
		S.xx_n = n;
	}
	ZG_LAUNCH(k_zds_finish, gm, 128, 0, s, archive, off, len, ulen, S.multi.as<u32>(), nmulti, S.tail.as<u64>(), S.f_out.as<u64>(),
	          S.f_status.as<u32>(), status, produced, cksums);
	ZG_COUNT_LAUNCH();
	if (zg_publish(s, totals + 2, h + 6, 8) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) return ZG_ERR(ZG_error_device);
	g_zd_stats[5] = h[6];
	return cudaGetLastError() == cudaSuccess ? 0 : ZG_ERR(ZG_error_device);
}

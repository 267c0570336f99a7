// Device helpers shared by the two Zstandard decode paths (RFC 8878; replaces DCtx::decompress_stream as driven by
// crates/zarc/src/decode/zstd_iterator.rs:88-153): the fused lane-per-frame kernel (zstd_decode.cu) and the staged
// pipeline for multi-block frames (zstd_decode_staged.cu).  Header and section parsers, Huffman / FSE table builds,
// the lane-private FSE sequence decoder and the row-wise sequence executor.
#pragma once
#include "common.h"
#include "zstd_common.cuh"

#define ZD_WARPS 4
#ifndef ZD_MIN_CTAS
#define ZD_MIN_CTAS 5                    // occupancy target: 20 warps / SM
#endif
#define ZD_SEQ_ARENA (1u << 17)          // u64 entries of sequence staging per warp (1 MiB)
#define ZD_LITBUF (ZS_BLOCK_MAX + 64)    // bytes of literal staging per warp
#define ZD_TAB_SLOT 1280u                // u32 entries per lane: LL 512 | ML 512 | OF 256
#define ZD_OFF_MAX ((1u << 28) - 1u)
#define ZD_BATCH_BYTES (128u << 10)        // least compressed bytes per warp batch (see the hand-out in the kernel)

struct ZdWarp {
	u32 tab[512];      // table under construction (FSE sequence table or Huffman-weight table)
	u16 huf[2048];     // sym | nbBits << 8
	u8 weights[256];   // Huffman weights (and, while FSE-coded ones are read, the list of nonzero counts)
	i16 norm[256];
	u16 next[256];     // FSE build scratch; Huffman: where each weight's table entries start
	u32 misc[8];
};

// flags
#define ZD_F_ACTIVE 1u      // frame still has blocks to decode
#define ZD_F_LAST 2u        // the block in flight is the frame's last
#define ZD_F_CKSUM 4u       // frame has a Content_Checksum
#define ZD_F_HUF_OK 8u      // a Huffman tree has been defined (ZdHufSave::tree is valid)
#define ZD_F_LL_OK 16u
#define ZD_F_ML_OK 32u
#define ZD_F_OF_OK 64u
#define ZD_F_LL_DEF 256u    // table = the predefined one (not in the slot)
#define ZD_F_ML_DEF 512u
#define ZD_F_OF_DEF 1024u
#define ZD_F_HAS_CK 2048u   // checksum field was read
#define ZD_F_LIT_STAGED 4096u  // the frame's Huffman literals were decoded ahead (k_zd_huf_literals); where: ZdHufSave::staged
#define ZD_F_LIT_BAD 8192u     // ... and found corrupt

// what a frame's Huffman literals leave for its later blocks; per lane of the fused kernel, in global scratch
struct ZdHufSave {
	const u8* tree;     // the description of the last tree the frame defined, for Treeless blocks (ZD_F_HUF_OK)
	const u8* staged;   // the literals k_zd_huf_literals decoded ahead (ZD_F_LIT_STAGED)
	u32 tree_n;         // the bytes the description may take
};

// the lane-private state of the FSE sequence decode (zd_lane_decode) of one block
struct ZdSeqState {
	ZsBack b;
	u32 sl, so, sm;     // the LL, OF and ML states
	u32 rep0, rep1, rep2;
	u32 left;           // sequences left
};

// one frame's decoding state; lives in the registers of the frame's lane
struct ZdLane {
	const u8* src;
	u8* out;
	u64 n, ip, cap, opos, fcs;
	u64 base;           // lowest output position a match may reach (0; the block's start for a split frame's block)
	u32 status, flags, fcs_len, cksum;
	u32 ll_log, ml_log, of_log;
	// block in flight
	const u8* blk;      // block body
	u32 blk_n;
	u32 nseq, seq_base;
	ZdSeqState seq;     // (the repeat offsets carry over from block to block)
};

template <typename T>
ZG_DEV T zd_bc(T v, int f) { return __shfl_sync(ZG_FULL, v, f); }
ZG_DEV const u8* zd_bc(const u8* v, int f) { return (const u8*)(uintptr_t)__shfl_sync(ZG_FULL, (u64)(uintptr_t)v, f); }
ZG_DEV u8* zd_bc(u8* v, int f) { return (u8*)(uintptr_t)__shfl_sync(ZG_FULL, (u64)(uintptr_t)v, f); }

// every lane gets a copy of lane f's frame state
ZG_DEV ZdLane zd_bcast(const ZdLane& L, int f) {
	ZdLane U;
	U.src = zd_bc(L.src, f);
	U.out = zd_bc(L.out, f);
	U.n = zd_bc(L.n, f);
	U.ip = zd_bc(L.ip, f);
	U.cap = zd_bc(L.cap, f);
	U.opos = zd_bc(L.opos, f);
	U.fcs = zd_bc(L.fcs, f);
	U.status = zd_bc(L.status, f);
	U.flags = zd_bc(L.flags, f);
	U.fcs_len = zd_bc(L.fcs_len, f);
	U.cksum = zd_bc(L.cksum, f);
	U.seq.rep0 = zd_bc(L.seq.rep0, f);
	U.seq.rep1 = zd_bc(L.seq.rep1, f);
	U.seq.rep2 = zd_bc(L.seq.rep2, f);
	U.ll_log = zd_bc(L.ll_log, f);
	U.ml_log = zd_bc(L.ml_log, f);
	U.of_log = zd_bc(L.of_log, f);
	U.base = zd_bc(L.base, f);
	U.blk = zd_bc(L.blk, f);
	U.blk_n = zd_bc(L.blk_n, f);
	U.nseq = zd_bc(L.nseq, f);
	U.seq.left = zd_bc(L.seq.left, f);
	U.seq_base = zd_bc(L.seq_base, f);
	U.seq.b.start = zd_bc(L.seq.b.start, f);
	U.seq.b.ptr = zd_bc(L.seq.b.ptr, f);
	U.seq.b.lo = zd_bc(L.seq.b.lo, f);
	U.seq.b.hi = zd_bc(L.seq.b.hi, f);
	U.seq.b.consumed = zd_bc(L.seq.b.consumed, f);
	U.seq.sl = zd_bc(L.seq.sl, f);
	U.seq.so = zd_bc(L.seq.so, f);
	U.seq.sm = zd_bc(L.seq.sm, f);
	return U;
}

// ---------------------------------------------------------------------------------------------
// Loads of bytes that ANOTHER SM may have written during this kernel (the staged pipeline's match sources: output of
// earlier blocks, executed by other warps) must not be served from this SM's L1: CG = ld.global.cg (L2 only).
template <bool CG>
ZG_DEV u32 zd_ldw(const u32* p) {
#ifndef ZG_EMU
	if (CG) return __ldcg(p);
#endif
	return *p;
}
template <bool CG>
ZG_DEV u32 zd_ldb(const u8* p) {
#ifndef ZG_EMU
	if (CG) return __ldcg(p);
#endif
	return *p;
}
// warp-cooperative copies
template <bool CG>
ZG_DEV_NOINLINE void zg_warp_copy_t(u8* dst, const u8* src, u32 n) {
	u32 lane = zg_lane();
	if (n < 128) {
		for (u32 i = lane; i < n; i += 32) dst[i] = (u8)zd_ldb<CG>(src + i);
		return;
	}
	u32 head = (u32)((16 - ((uintptr_t)dst & 15)) & 15);
	if (lane < head) dst[lane] = (u8)zd_ldb<CG>(src + lane);
	dst += head;
	src += head;
	n -= head;
	u32 nvec = n >> 4;
	uintptr_t sa = (uintptr_t)src;
	const u32* sw = (const u32*)(sa & ~(uintptr_t)3);
	u32 sh = (u32)(sa & 3) * 8;
	for (u32 v = lane; v < nvec; v += 32) {
		const u32* q = sw + 4 * v;
		u32 w0 = zd_ldw<CG>(q), w1 = zd_ldw<CG>(q + 1), w2 = zd_ldw<CG>(q + 2), w3 = zd_ldw<CG>(q + 3);
		uint4 o;
		if (sh == 0) {
			o = make_uint4(w0, w1, w2, w3);
		} else {
			u32 w4 = zd_ldw<CG>(q + 4);
			o = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
			               __funnelshift_r(w3, w4, sh));
		}
		((uint4*)dst)[v] = o;
	}
	for (u32 i = (nvec << 4) + lane; i < n; i += 32) dst[i] = (u8)zd_ldb<CG>(src + i);
}
ZG_DEV void zg_warp_copy(u8* dst, const u8* src, u32 n) { zg_warp_copy_t<false>(dst, src, n); }
ZG_DEV_NOINLINE void zg_warp_fill(u8* dst, u32 byte, u32 n) {
	for (u32 i = zg_lane(); i < n; i += 32) dst[i] = (u8)byte;
}
// match copy inside the frame output: d[i] = d[i - off], forward semantics (overlap allowed)
template <bool CG>
ZG_DEV void zd_warp_match(u8* d, u32 off, u32 ml) {
	u32 lane = zg_lane();
	const u8* s = d - off;
	if (off >= 32) {
		bool overlap = off < ml;
		for (u32 i0 = 0; i0 < ml; i0 += 32) {
			u32 i = i0 + lane;
			if (i < ml) d[i] = (u8)zd_ldb<CG>(s + i);
			if (overlap) __syncwarp();
		}
	} else {
		for (u32 i = lane; i < ml; i += 32) d[i] = (u8)zd_ldb<CG>(s + i % off);
	}
}

// ---------------------------------------------------------------------------------------------
// Huffman tree descriptions (RFC 8878 §4.2.1), each read on one lane (zd_read_huf_weights_lane, zd_huf_weights_check):
// by lane 0 of the warp that decodes the block (zd_warp_huf_literals), or one per lane in k_zd_huf_literals.  The
// table is then filled warp-wide (zd_huf_fill_table).

// The description's size from its header byte: direct weights (*nw of them, as nibbles) or FSE-coded (*nw = 0).
// Returns the bytes it takes (0 when they do not fit in n, or an FSE description is shorter than 2 bytes).
ZG_DEV u32 zd_huf_desc_size(const u8* src, u32 n, u32* nw) {
	if (n < 1) return 0;
	u32 h = src[0];
	*nw = h >= 128 ? h - 127 : 0;
	u32 used = h >= 128 ? 1 + ((h - 126) >> 1) : 1 + h;
	return used > n || h < 2 ? 0 : used;
}
ZG_DEV void zd_huf_direct_weights(const u8* src, u32 i, u8* weights) {
	u32 byte = src[1 + (i >> 1)];
	weights[i] = (u8)((i & 1) ? (byte & 15) : (byte >> 4));
}
// FSE-coded weights after the NCount: two interleaved states; when the stream runs dry after an update, the other
// state's symbol is the last one (RFC 8878 §4.2.1.2).  Returns how many (0 on error).  Single thread.
ZG_DEV u32 zd_huf_fse_weights(const u32* tab, u32 log, const u8* src, u32 n, u8* weights) {
	ZsBack b;
	if (!zs_back_init(b, src, n)) return 0;
	u32 cnt = 0;
	zs_back_reload(b);
	u32 s1 = zs_back_read(b, log), s2 = zs_back_read(b, log);
	for (;;) {
		if (cnt > 253) return 0;
		u32 e1 = tab[s1];
		weights[cnt++] = (u8)e1;
		zs_back_reload(b);
		s1 = (e1 >> 16) + zs_back_read(b, (e1 >> 8) & 0xff);
		if (zs_back_overflow(b)) {
			weights[cnt++] = (u8)tab[s2];
			return cnt;
		}
		u32 e2 = tab[s2];
		weights[cnt++] = (u8)e2;
		s2 = (e2 >> 16) + zs_back_read(b, (e2 >> 8) & 0xff);
		if (zs_back_overflow(b)) {
			weights[cnt++] = (u8)tab[s1];
			return cnt;
		}
	}
}
// The checks of a tree given its explicit weights (all <= 11) as their sum of 2^(w-1) and how many are 1: returns
// maxbits (0 when the tree is invalid) and sets the implied last weight.
ZG_DEV u32 zd_huf_tree_check(u32 sum, u32 ones, u32& last) {
	if (sum == 0) return 0;
	u32 maxbits = zs_highbit(sum) + 1;
	u32 left = (1u << maxbits) - sum;
	if (maxbits > ZS_HUF_MAXLOG || (left & (left - 1))) return 0;
	last = zs_highbit(left) + 1;
	ones += last == 1;
	if (ones < 2 || (ones & 1)) return 0;  // as libzstd HUF_readStats
	return maxbits;
}
// A tree description -> weights[0..nw) (the last weight is implied).  Returns the bytes it takes (0 on error).  `fse`
// (64 cells) and `list` (64 words, which may be `weights` itself) are the lane's scratch for FSE-coded weights.
ZG_DEV u32 zd_read_huf_weights_lane(const u8* src, u32 n, u8* weights, u32* fse, u32* list, u32* nw_out) {
	u32 nw;
	u32 used = zd_huf_desc_size(src, n, &nw);
	if (used == 0) return 0;
	if (nw) {
		for (u32 i = 0; i < nw; i++) zd_huf_direct_weights(src, i, weights);
	} else {
		u32 csz = used - 1, nsym = 0, log = 0, ne = 0;
		// the symbols with a nonzero count: at most 1 << log of them (each takes at least one of the cells).  Symbols
		// above 11 may be declared; a weight above 11 is only an error when it is decoded (zd_huf_tree_check's caller)
		u32 nc = zs_read_ncount_to(src + 1, csz, 6, 255, [&](u32 s, i32 v) { if (v) list[ne++] = ZS_FSE_ENTRY(s, v); }, &nsym, &log);
		if (nc == 0 || nc >= csz) return 0;
		zs_fse_build_dtable_lane(fse, list, ne, log);
		nw = zd_huf_fse_weights(fse, log, src + 1 + nc, csz - nc, weights);
		if (nw == 0) return 0;
	}
	*nw_out = nw;
	return used;
}

// weights[0..nw) -> maxbits (0 when the tree is invalid), the implied last weight at weights[nw], and where each
// weight's entries start in the table: start[w] for w = 1..11.  Single thread: the counts per weight are kept in
// registers, as 10-bit fields (three weights per word).
ZG_DEV u32 zd_huf_weights_check(u8* weights, u32 nw, u16* start) {
	u32 c0 = 0, c1 = 0, c2 = 0, c3 = 0;
	bool ok = true;
	for (u32 i = 0; i < nw; i++) {
		u32 w = weights[i];
		ok &= w <= 11;
		u32 q = (w * 11) >> 5, inc = w <= 11 ? 1u << ((w - 3 * q) * 10) : 0;  // (q = w / 3 for w <= 11)
		c0 += q == 0 ? inc : 0;
		c1 += q == 1 ? inc : 0;
		c2 += q == 2 ? inc : 0;
		c3 += q == 3 ? inc : 0;
	}
	auto count = [&](u32 w) { return ((w < 3 ? c0 : w < 6 ? c1 : w < 9 ? c2 : c3) >> ((w % 3) * 10)) & 1023u; };
	u32 sum = 0, last = 0;
	ZG_UNROLL
	for (u32 w = 1; w <= 11; w++) sum += count(w) << (w - 1);
	u32 maxbits = ok ? zd_huf_tree_check(sum, count(1), last) : 0;
	if (maxbits == 0) return 0;
	weights[nw] = (u8)last;
	u32 at = 0;
	ZG_UNROLL
	for (u32 w = 1; w <= 11; w++) {
		start[w] = (u16)at;
		at += (count(w) + (w == last)) << (w - 1);
	}
	return maxbits;
}

// weights[0..nsym) -> huf (1 << maxbits entries), all in shared memory: the symbols of weight w take 2^(w-1) entries
// each, in symbol order from start[w] on (zd_huf_weights_check; start[w] is advanced).  A symbol's start is its weight's
// plus the entries of the symbols of that weight before it (match_any over 32 symbols at a time).  Short ranges are
// written by the owning lane, long ones by the warp.  All lanes call.
ZG_DEV void zd_huf_fill_table(u16* huf, const u8* weights, u32 nsym, u16* start, u32 maxbits) {
	u32 lane = zg_lane();
	for (u32 s0 = 0; s0 < nsym; s0 += 32) {
		u32 s = s0 + lane, w = s < nsym ? weights[s] : 0;
		u32 peers = __match_any_sync(ZG_FULL, w);
		u32 len = w ? 1u << (w - 1) : 0;
		u32 at = w ? start[w] + (u32)__popc(peers & zg_lanemask_lt()) * len : 0;
		__syncwarp();
		if (w && (peers & zg_lanemask_lt()) == 0) start[w] += (u32)__popc(peers) * len;
		u32 entry = s | ((maxbits + 1 - w) << 8);
		if (len > 0 && len < 32)
			for (u32 k = 0; k < len; k++) huf[at + k] = (u16)entry;
		u32 big = __ballot_sync(ZG_FULL, len >= 32);
		while (big) {
			int l = __ffs((int)big) - 1;
			big &= big - 1;
			u32 bs = __shfl_sync(ZG_FULL, at, l), bl = __shfl_sync(ZG_FULL, len, l), be = __shfl_sync(ZG_FULL, entry, l);
			for (u32 k = lane; k < bl; k += 32) huf[bs + k] = (u16)be;
		}
		__syncwarp();
	}
}

// one Huffman stream, single thread.  Four symbols per refill of the bit container, stored as one aligned word (byte
// stores up to the first 4-byte boundary of dst and at the end): lanes decoding different streams write to different
// lines, so every store instruction costs the memory system one request per lane.
ZG_DEV_NOINLINE bool zd_huf_stream(const u16* huf, u32 maxbits, const u8* src, u32 n, u8* dst, u32 count) {
	ZsBack b;
	if (!zs_back_init(b, src, n)) return false;
	u32 i = 0;
	const u32 sh = 32u - maxbits;
	const u32 head = zg_min<u32>(count, (u32)(0u - (uintptr_t)dst) & 3u);
	while (i < count) {
		zs_back_reload(b);
		u32 m = i < head ? head - i : zg_min<u32>(count - i, 4u);  // 4 x 11 bits <= 57
		// the unread bits left-aligned in ah:al; every symbol then costs one shift for the index and a two-word
		// shift for the bits it used (bits before the start of the stream shift in as zeros)
		u32 c = b.consumed;
		u32 ah = c < 32 ? __funnelshift_l(b.lo, b.hi, c) : (c < 64 ? b.lo << (c & 31u) : 0u);
		u32 al = c < 32 ? b.lo << c : 0u;
		u32 used = 0, word = 0;
		for (u32 k = 0; k < m; k++) {
			u32 e = huf[ah >> sh];
			word |= (e & 0xffu) << (8 * k);
			u32 nb = e >> 8;
			ah = __funnelshift_l(al, ah, nb);
			al <<= nb;
			used += nb;
		}
		if (m == 4) *(u32*)(dst + i) = word;
		else
			for (u32 k = 0; k < m; k++) dst[i + k] = (u8)(word >> (8 * k));
		b.consumed = c + used;
		i += m;
	}
	zs_back_reload(b);
	return zs_back_finished(b);
}

// Where stream j of a Huffman literals section lies: lp..lend = the streams (after the tree description), `streams`
// 1 or 4 (a 4-stream section starts with its jump table).  Sets the stream's bytes, its first literal and its count
// (0 streams past the section's count).  Returns false on a bad jump table.
ZG_DEV bool zd_huf_split(const u8* lp, const u8* lend, u32 regen, u32 streams, u32 j, const u8*& sp, u32& sn, u32& first, u32& cnt) {
	if (streams == 1) {
		sp = lp;
		sn = (u32)(lend - lp);
		first = 0;
		cnt = j == 0 ? regen : 0;
		return true;
	}
	if (lend - lp < 10) return false;
	u32 s1 = zg_ld16(lp), s2 = zg_ld16(lp + 2), s3 = zg_ld16(lp + 4);
	lp += 6;
	u32 avail = (u32)(lend - lp);
	u32 seg = (regen + 3) >> 2;
	if (s1 + s2 + s3 >= avail || seg * 3 > regen) return false;
	u32 so = j == 0 ? 0 : j == 1 ? s1 : j == 2 ? s1 + s2 : s1 + s2 + s3;
	sn = j == 0 ? s1 : j == 1 ? s2 : j == 2 ? s3 : avail - s1 - s2 - s3;
	sp = lp + so;
	first = j * seg;
	cnt = j < 3 ? seg : regen - 3 * seg;
	return true;
}

// sequence table for one of LL/OF/ML into the lane's global slot `slot`.  All lanes call (uniform).
// Returns false on error; advances p.  `flags`: def_flag is set when the predefined table is in use.
ZG_DEV_NOINLINE bool zd_seq_table(ZdWarp* W, u32* slot, u32& log, u32& flags, u32 ok_flag, u32 def_flag, u32 mode, const u8*& p, const u8* end,
                         u32 maxlog, u32 maxsym, u32 def_log) {
	u32 lane = zg_lane();
	if (mode == 0) {
		log = def_log;
		flags |= ok_flag | def_flag;
		return true;
	}
	if (mode == 1) {
		if (p >= end) return false;
		u32 sym = *p++;
		if (sym > maxsym) return false;
		if (lane == 0) slot[0] = sym;
		log = 0;
		flags = (flags | ok_flag) & ~def_flag;
		return true;
	}
	if (mode == 2) {
		if (lane == 0) {
			u32 nsym = 0, lg = 0;
			u32 nc = zs_read_ncount(p, (u32)(end - p), maxlog, maxsym, W->norm, &nsym, &lg);
			W->misc[0] = nc;
			W->misc[1] = nsym;
			W->misc[2] = lg;
		}
		__syncwarp();
		u32 nc = W->misc[0], nsym = W->misc[1], lg = W->misc[2];
		__syncwarp();
		if (nc == 0) return false;
		zs_fse_build_dtable(W->tab, W->norm, nsym, lg, W->next);
		for (u32 i = lane; i < (1u << lg); i += 32) slot[i] = W->tab[i];
		__syncwarp();
		p += nc;
		log = lg;
		flags = (flags | ok_flag) & ~def_flag;
		return true;
	}
	return (flags & ok_flag) != 0;  // Repeat_Mode: the slot (or the predefined flag) still holds the table
}

// The sequences bitstream p..end of a block and the three initial states.  Returns false when malformed.
ZG_DEV bool zd_seq_start(ZdSeqState& s, const u8* p, const u8* end, u32 ll_log, u32 of_log, u32 ml_log) {
	if (!zs_back_init(s.b, p, (u32)(end - p))) return false;
	zs_back_reload(s.b);
	s.sl = zs_back_read(s.b, ll_log);
	s.so = zs_back_read(s.b, of_log);
	s.sm = zs_back_read(s.b, ml_log);
	return !zs_back_overflow(s.b);
}

// ---------------------------------------------------------------------------------------------
ZG_DEV void zd_fail(ZdLane& U, u32 code) {
	U.status = code;
	U.flags &= ~ZD_F_ACTIVE;
	U.nseq = U.seq.left = 0;
}
// end of frame: optional checksum field, content-size check
ZG_DEV void zd_frame_finish(ZdLane& U) {
	U.flags &= ~ZD_F_ACTIVE;
	U.nseq = U.seq.left = 0;
	if (U.flags & ZD_F_CKSUM) {
		if (U.ip + 4 > U.n) {
			U.status = ZS_E_SRC_SIZE;
			return;
		}
		U.cksum = zg_ld32(U.src + U.ip);
		U.flags |= ZD_F_HAS_CK;
		U.ip += 4;
	}
	if (U.fcs_len && U.fcs != U.opos) U.status = ZS_E_CORRUPT;
}

// Frame_Header (RFC 8878 §3.1.1.1) of the frame src[0..n): where its first block starts, the content size (fcs_len
// bytes of it were given, 0: none) and whether a Content_Checksum ends the frame (all 0 when the header is bad).
// Returns a ZS_E_* code.  Single thread.
struct ZdFrameHdr {
	u64 ip, fcs;
	u32 fcs_len, cksum;
};
ZG_DEV u32 zd_frame_header(const u8* src, u64 n, ZdFrameHdr& F) {
	F.ip = F.fcs = 0;
	F.fcs_len = F.cksum = 0;
	if (n < 6) return ZS_E_SRC_SIZE;
	if (zg_ld32(src) != ZS_MAGIC) return ZS_E_PREFIX;
	u32 desc = src[4];
	u32 fcs_flag = desc >> 6, single = (desc >> 5) & 1, checksum = (desc >> 2) & 1, did_flag = desc & 3;
	if (desc & 8) return ZS_E_UNSUPPORTED;
	u64 ip = 5;
	u64 window = 0;
	if (!single) {
		u32 wd = src[ip++];
		u32 wl = 10 + (wd >> 3);
		if (wl > 31) return ZS_E_WINDOW;
		window = ((u64)1 << wl) + ((((u64)1 << wl) >> 3) * (wd & 7));
	}
	if (did_flag) {
		u32 dl = did_flag == 3 ? 4 : did_flag;
		if (ip + dl > n) return ZS_E_SRC_SIZE;
		u32 did = 0;
		for (u32 i = 0; i < dl; i++) did |= (u32)src[ip + i] << (8 * i);
		ip += dl;
		if (did) return ZS_E_DICT;
	}
	u32 fcs_len = fcs_flag == 0 ? single : fcs_flag == 1 ? 2 : fcs_flag == 2 ? 4 : 8;
	if (ip + fcs_len > n) return ZS_E_SRC_SIZE;
	u64 fcs = 0;
	for (u32 i = 0; i < fcs_len; i++) fcs |= (u64)src[ip + i] << (8 * i);
	if (fcs_len == 2) fcs += 256;
	ip += fcs_len;
	// libzstd's streaming decoder (what zstd_iterator.rs:29 creates) refuses windows > 2^27
	// ("Frame requires too much memory for decoding", SURVEY.md App. C)
	if ((single ? fcs : window) > ((u64)1 << 27)) return ZS_E_WINDOW;
	F.ip = ip;
	F.fcs = fcs;
	F.fcs_len = fcs_len;
	F.cksum = checksum;
	return ZS_OK;
}

// ---------------------------------------------------------------------------------------------
// Literals_Section_Header (RFC 8878 §3.1.1.3.1.1).  Returns false on a malformed header.
struct ZdLitHdr {
	u32 ltype, regen, comp, hdr, streams;
};
ZG_DEV bool zd_lit_header(const u8* src, u32 n, ZdLitHdr& h) {
	if (n < 2) return false;
	u32 b0 = src[0];
	u32 sf = (b0 >> 2) & 3;
	h.ltype = b0 & 3;
	h.comp = 0;
	h.streams = 1;
	if (h.ltype < 2) {
		if (sf == 0 || sf == 2) {
			h.regen = b0 >> 3;
			h.hdr = 1;
		} else if (sf == 1) {
			h.regen = (b0 >> 4) | ((u32)src[1] << 4);
			h.hdr = 2;
		} else {
			if (n < 3) return false;
			h.regen = (b0 >> 4) | ((u32)src[1] << 4) | ((u32)src[2] << 12);
			h.hdr = 3;
		}
		if (h.regen > ZS_BLOCK_MAX) return false;
		h.comp = h.ltype == 0 ? h.regen : 1;
		return h.hdr + h.comp <= n;
	}
	if (n < 3) return false;
	u64 v = (u64)b0 | ((u64)src[1] << 8) | ((u64)src[2] << 16);
	if (sf == 0 || sf == 1) {
		h.regen = (u32)(v >> 4) & 1023;
		h.comp = (u32)(v >> 14) & 1023;
		h.hdr = 3;
		h.streams = sf == 0 ? 1 : 4;
	} else if (sf == 2) {
		if (n < 4) return false;
		v |= (u64)src[3] << 24;
		h.regen = (u32)(v >> 4) & 16383;
		h.comp = (u32)(v >> 18) & 16383;
		h.hdr = 4;
		h.streams = 4;
	} else {
		if (n < 5) return false;
		v |= ((u64)src[3] << 24) | ((u64)src[4] << 32);
		h.regen = (u32)(v >> 4) & 262143;
		h.comp = (u32)(v >> 22) & 262143;
		h.hdr = 5;
		h.streams = 4;
	}
	return h.regen <= ZS_BLOCK_MAX && h.hdr + h.comp <= n && h.regen != 0;
}

// The literals section of a single-block frame when it is Huffman-coded with a fresh tree (type 2), the only kind
// k_zd_huf_literals decodes ahead: its archive offset and Regenerated_Size.  Reads the headers exactly as the fused
// kernel does; anything it cannot take (other literal types, more blocks, bad headers) is left to the fused kernel.
#define ZD_LIT_NONE (~0ull)        // lit_at[k]: not decoded ahead
#define ZD_LIT_BAD (~0ull - 1ull)  // ... decoded ahead and corrupt
ZG_DEV bool zd_single_huf_section(const u8* archive, u64 archive_len, u64 fo, u64 fl, u64& at, u32& regen) {
	if (fo > archive_len || fl > archive_len - fo) return false;
	const u8* src = archive + fo;
	ZdFrameHdr F;
	if (zd_frame_header(src, fl, F) != ZS_OK || F.ip + 3 > fl) return false;
	u32 bh = zg_ld24(src + F.ip), bsize = bh >> 3;
	if ((bh & 7u) != 5u || bsize > ZS_BLOCK_MAX || F.ip + 3 + bsize > fl) return false;  // Last_Block, Compressed_Block
	ZdLitHdr h;
	if (!zd_lit_header(src + F.ip + 3, bsize, h) || h.ltype != 2) return false;
	at = fo + F.ip + 3;
	regen = h.regen;
	return true;
}

// Literals_Section_Header and Sequences_Section_Header of a compressed block (RFC 8878 §3.1.1.3): Number_of_Sequences
// (at most `maxseq`) and Symbol_Compression_Modes.  Returns false when malformed.  Single thread.
struct ZdSect {
	ZdLitHdr h;
	u32 nseq, modes;
	const u8* tables;   // first table description (after the modes byte)
};
ZG_DEV bool zd_sections(const u8* src, u32 n, u32 maxseq, ZdSect& S) {
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
	return (S.modes & 3) == 0 && S.nseq <= maxseq;
}

// Huffman literals of one block (uniform in the warp) into dst: lp = the section after its header, `tree` / `tn` = the
// tree description and the bytes it may take (for a Huffman_Literals_Block its own, at lp; for a Treeless one the
// description of the block that last defined a tree).  Lane 0 reads the tree.  Returns a ZS_E_* code.
ZG_DEV_NOINLINE u32 zd_warp_huf_literals(ZdWarp* W, const u8* tree, u32 tn, const u8* lp, const ZdLitHdr& h, u8* dst) {
	u32 lane = zg_lane();
	u32 used = 0, nw = 0, bits = 0;
	if (lane == 0) {
		used = zd_read_huf_weights_lane(tree, tn, W->weights, W->tab, (u32*)W->weights, &nw);
		bits = used ? zd_huf_weights_check(W->weights, nw, W->next) : 0;
	}
	__syncwarp();
	bits = __shfl_sync(ZG_FULL, bits, 0);
	if (bits == 0) return ZS_E_CORRUPT;
	used = __shfl_sync(ZG_FULL, used, 0);
	nw = __shfl_sync(ZG_FULL, nw, 0);
	zd_huf_fill_table(W->huf, W->weights, nw + 1, W->next, bits);
	const u8* lend = lp + h.comp;
	if (h.ltype == 2) lp += used;
	const u8* sp;
	u32 sn, first, cnt;
	if (!zd_huf_split(lp, lend, h.regen, h.streams, lane, sp, sn, first, cnt)) return ZS_E_CORRUPT;
	bool ok = true;
	if (lane < h.streams) ok = zd_huf_stream(W->huf, bits, sp, sn, dst + first, cnt);
	if (!__all_sync(ZG_FULL, ok)) return ZS_E_CORRUPT;
	__syncwarp();
	return ZS_OK;
}

// The block's literals (uniform in the warp): Raw -> pointer into the block, RLE -> the byte,
// Huffman -> decoded into litbuf.  Returns a ZS_E_* code.
ZG_DEV_NOINLINE u32 zd_literals(ZdWarp* W, u32& flags, const u8* src, const ZdLitHdr& h, u8* litbuf, ZdHufSave* save, const u8*& lit,
                       bool& lit_rle, u32& rle_byte) {
	lit_rle = false;
	rle_byte = 0;
	if (h.ltype == 0) {
		lit = src + h.hdr;
		return ZS_OK;
	}
	if (h.ltype == 1) {
		lit_rle = true;
		rle_byte = src[h.hdr];
		lit = src;
		return ZS_OK;
	}
	if (flags & (ZD_F_LIT_STAGED | ZD_F_LIT_BAD)) {  // a single-block frame's literals, decoded ahead by k_zd_huf_literals
		if (flags & ZD_F_LIT_BAD) return ZS_E_CORRUPT;
		flags |= ZD_F_HUF_OK;
		lit = save->staged;
		return ZS_OK;
	}
	const u8* lp = src + h.hdr;
	const u8* tree = lp;
	u32 tn = h.comp;
	if (h.ltype == 2) {  // a later Treeless block reads this description again
		if (zg_lane() == 0) {
			save->tree = lp;
			save->tree_n = h.comp;
		}
	} else {
		if (!(flags & ZD_F_HUF_OK)) return ZS_E_CORRUPT;
		tree = save->tree;
		tn = save->tree_n;
	}
	u32 r = zd_warp_huf_literals(W, tree, tn, lp, h, litbuf);
	if (r) return r;
	flags |= ZD_F_HUF_OK;
	lit = litbuf;
	return ZS_OK;
}

// ---------------------------------------------------------------------------------------------
// Phase A for one Compressed block of the frame viewed by U (uniform in the warp).  Returns 0 = ok
// (U.nseq sequences wait for phase B; 0 means the block was literals only and is complete),
// ZD_DEFER = the sequence arena is full (nothing consumed), else a ZS_E_* code + 1.
#define ZD_DEFER 1u
#define ZD_ERR(c) ((c) + 1u)
// The emulator build counts scheduling events no output shows, so that its tests can prove which ones a batch reached:
// [0] block set-ups deferred for arena space, [1] rounds of the Huffman literals pre-pass (zg_internal_sched_stats).
// The product build has no counter.
#ifdef ZG_EMU
extern u64 g_zd_sched[2];
#define ZD_SCHED_COUNT(i) (zg_lane() == 0 ? (void)g_zd_sched[i]++ : (void)0)
#else
#define ZD_SCHED_COUNT(i) ((void)0)
#endif
ZG_DEV u32 zd_block_setup(ZdWarp* W, ZdLane& U, const u8* src, u32 n, u32* slot, u32& arena_used, u8* litbuf, ZdHufSave* save) {
	ZdSect S;
	// (the arena bounds the count: > 131072 sequences cannot come from a 128 KiB block)
	if (!zd_sections(src, n, ZD_SEQ_ARENA, S)) return ZD_ERR(ZS_E_CORRUPT);
	const ZdLitHdr& h = S.h;
	if (S.nseq == 0) {
		const u8* lit;
		bool lit_rle;
		u32 rle_byte;
		u32 r = zd_literals(W, U.flags, src, h, litbuf, save, lit, lit_rle, rle_byte);
		if (r) return ZD_ERR(r);
		if (U.opos + h.regen > U.cap) return ZD_ERR(ZS_E_DST_SMALL);
		if (h.regen) {
			if (lit_rle) zg_warp_fill(U.out + U.opos, rle_byte, h.regen);
			else zg_warp_copy(U.out + U.opos, lit, h.regen);
		}
		U.opos += h.regen;
		U.nseq = U.seq.left = 0;
		__syncwarp();
		return 0;
	}
	if (arena_used + S.nseq > ZD_SEQ_ARENA) {  // (an empty arena always fits a block)
		ZD_SCHED_COUNT(0);
		return ZD_DEFER;
	}
	const u8* end = src + n;
	const u8* p = S.tables;
	u32 modes = S.modes;
	if (!zd_seq_table(W, slot, U.ll_log, U.flags, ZD_F_LL_OK, ZD_F_LL_DEF, (modes >> 6) & 3, p, end, ZS_LL_MAXLOG, 35, 6)) return ZD_ERR(ZS_E_CORRUPT);
	if (!zd_seq_table(W, slot + 1024, U.of_log, U.flags, ZD_F_OF_OK, ZD_F_OF_DEF, (modes >> 4) & 3, p, end, ZS_OF_MAXLOG, 31, 5)) return ZD_ERR(ZS_E_CORRUPT);
	if (!zd_seq_table(W, slot + 512, U.ml_log, U.flags, ZD_F_ML_OK, ZD_F_ML_DEF, (modes >> 2) & 3, p, end, ZS_ML_MAXLOG, 52, 6)) return ZD_ERR(ZS_E_CORRUPT);
	// (uniform here; the frame's lane keeps the state)
	if (!zd_seq_start(U.seq, p, end, U.ll_log, U.of_log, U.ml_log)) return ZD_ERR(ZS_E_CORRUPT);
	U.nseq = U.seq.left = S.nseq;
	U.seq_base = arena_used;
	U.blk = src;
	U.blk_n = n;
	arena_used += S.nseq;
	__syncwarp();
	return 0;
}

// Advance the frame viewed by U (uniform) through its blocks until one with sequences is ready for
// phase B, the frame ends, fails, or has to wait for arena space.
ZG_DEV void zd_setup_frame(ZdWarp* W, ZdLane& U, u32* slot, u32& arena_used, u8* litbuf, ZdHufSave* save) {
	for (;;) {
		if (U.ip + 3 > U.n) return zd_fail(U, ZS_E_SRC_SIZE);
		u32 bh = zg_ld24(U.src + U.ip);
		u32 last = bh & 1, type = (bh >> 1) & 3, bsize = bh >> 3;
		if (type == 3) return zd_fail(U, ZS_E_CORRUPT);
		u64 body = U.ip + 3;
		if (type == 0) {
			if (body + bsize > U.n) return zd_fail(U, ZS_E_SRC_SIZE);
			if (bsize > ZS_BLOCK_MAX) return zd_fail(U, ZS_E_CORRUPT);
			if (U.opos + bsize > U.cap) return zd_fail(U, ZS_E_DST_SMALL);
			zg_warp_copy(U.out + U.opos, U.src + body, bsize);
			U.opos += bsize;
			U.ip = body + bsize;
		} else if (type == 1) {
			if (body + 1 > U.n) return zd_fail(U, ZS_E_SRC_SIZE);
			if (bsize > ZS_BLOCK_MAX) return zd_fail(U, ZS_E_CORRUPT);
			if (U.opos + bsize > U.cap) return zd_fail(U, ZS_E_DST_SMALL);
			zg_warp_fill(U.out + U.opos, U.src[body], bsize);
			U.opos += bsize;
			U.ip = body + 1;
		} else {
			if (bsize > ZS_BLOCK_MAX) return zd_fail(U, ZS_E_CORRUPT);
			if (body + bsize > U.n) return zd_fail(U, ZS_E_SRC_SIZE);
			u32 r = zd_block_setup(W, U, U.src + body, bsize, slot, arena_used, litbuf, save);
			if (r == ZD_DEFER) return;
			if (r) return zd_fail(U, r - 1u);
			U.ip = body + bsize;
			if (U.nseq) {
				U.flags = last ? (U.flags | ZD_F_LAST) : (U.flags & ~ZD_F_LAST);
				return;
			}
		}
		__syncwarp();
		if (last) return zd_frame_finish(U);
	}
}

// ---------------------------------------------------------------------------------------------
// The fused kernel's policy for zd_lane_decode: offsets beyond 2^28 exceed every window this decoder accepts; an
// offset of 0 only arises from a corrupt stream or from the unknown repeat-offset history of a split frame's block (then
// the block is not independent); lengths are < 2^18 by construction.  No bookkeeping.
struct ZdSeqPlain {
	static ZG_DEV bool bad(u32 off, bool) { return off - 1u >= ZD_OFF_MAX; }
	ZG_DEV void seq(u32, u32, u32) {}
};

// Phase B, lane-private: decode up to `cnt` sequences of this lane's block and append them, packed
// (offset:28 | litLength:18 | matchLength:18), to dst.  The caller keeps all lanes in step (cnt is bounded) so that the
// warp stays converged.  POL::bad(off, fresh) checks an offset (fresh: not a repeat code), P.seq(off, ll, ml) follows
// every sequence.  S and P are written back only when the call succeeds.
template <class POL>
ZG_DEV bool zd_lane_decode(ZdSeqState& S, POL& P, u32 cnt, const u32* llt, const u32* mlt, const u32* oft, u64* dst) {
	ZsBack b = S.b;
	u32 sl = S.sl, so = S.so, sm = S.sm;
	u32 rep0 = S.rep0, rep1 = S.rep1, rep2 = S.rep2;
	u32 left = S.left;
	POL pol = P;
	ZsBelow ahead = {0, 0};
	zs_below_fetch(b, ahead);
	u32 bad = 0;  // checked once per call: a bad sequence only poisons values, never an address (states stay inside their tables)
	for (u32 k = 0; k < cnt; k++) {
		u32 oe = oft[so], me = mlt[sm], le = llt[sl];
		zs_back_reload_ahead(b, ahead);  // >= 57 bits available from here; no memory wait (the bytes came in a step ago)
		// the codes come out of tables whose symbols were range-checked when they were read (zd_seq_table)
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
			if (used > 30) zs_back_reload_ahead(b, ahead);  // the three state updates need <= 26 bits
			sl = (le >> 16) + zs_back_read(b, (le >> 8) & 0xff);
			sm = (me >> 16) + zs_back_read(b, (me >> 8) & 0xff);
			so = (oe >> 16) + zs_back_read(b, (oe >> 8) & 0xff);
		}
		// repeat-offset resolution (RFC 8878 §3.1.1.5)
		u32 off;
		if (ofv > 3) {
			off = ofv - 3;
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
		}
		bad |= POL::bad(off, ofv > 3) ? 1u : 0u;
		pol.seq(off, ll, ml);
		dst[k] = (u64)off | ((u64)ll << 28) | ((u64)ml << 46);
	}
	if (bad || zs_back_overflow(b)) return false;
	left -= cnt;
	if (left == 0) {
		zs_back_reload(b);
		if (!zs_back_finished(b)) return false;
	}
	S.b = b;
	S.sl = sl;
	S.so = so;
	S.sm = sm;
	S.rep0 = rep0;
	S.rep1 = rep1;
	S.rep2 = rep2;
	S.left = left;
	P = pol;
	return true;
}

// Per-lane copy of n bytes between regions that do not overlap: 16 bytes per memory round trip (the
// loads of a group are all in flight before the first store).  Only aligned words that hold at least
// one source byte are touched.
template <bool CG>
ZG_DEV void zd_lane_copy(u8* dst, const u8* src, u32 n) {
	const u8* lim = src + n;
	for (u32 k0 = 0; k0 < n; k0 += 16) {
		uintptr_t a = (uintptr_t)(src + k0);
		const u32* w = (const u32*)(a & ~(uintptr_t)3);
		u32 sh = (u32)(a & 3) * 8;
		u32 x[5];
		ZG_UNROLL
		for (int k = 0; k < 5; k++) x[k] = (const u8*)(w + k) < lim ? zd_ldw<CG>(w + k) : 0u;
		u32 m = n - k0;
		u8* q = dst + k0;
		ZG_UNROLL
		for (int j = 0; j < 4; j++) {
			if (4u * j < m) {
				u32 v = __funnelshift_r(x[j], x[j + 1], sh);
				q[4 * j] = (u8)v;
				if (4u * j + 1 < m) q[4 * j + 1] = (u8)(v >> 8);
				if (4u * j + 2 < m) q[4 * j + 2] = (u8)(v >> 16);
				if (4u * j + 3 < m) q[4 * j + 3] = (u8)(v >> 24);
			}
		}
	}
}
// Per-lane match copy d[i] = d[i - off] for off < ml (the match overlaps its own output): the valid
// span [d - off, d + done) is periodic in `off`, so it is extended by non-overlapping copies whose
// length doubles.
template <bool CG>
ZG_DEV void zd_lane_overlap(u8* d, u32 off, u32 ml) {
	u32 done = 0;
	while (done < ml) {
		u32 c = zg_min<u32>(done + off, ml - done);
		zd_lane_copy<CG>(d + done, d - off, c);
		done += c;
	}
}

#ifndef ZD_LANE_COPY_MAX
#define ZD_LANE_COPY_MAX 64u   // longer literal runs / matches are copied by the whole warp
#endif

// Phase C: execute `cnt` (<= 32) sequences, one per lane.  Output and literal positions come from
// warp scans.  All literal runs are independent and copied first, lane-parallel.  Matches then go in
// waves: a match is ready once every earlier match of the row whose output its source overlaps has been
// written (match starts and ends grow with the lane, so that set is a range of lanes, found by two binary
// searches over shuffles); all ready matches of a wave copy lane-parallel.  A row of n sequences takes (dependency depth) waves, not n
// steps, and every wave is a few 16-byte round trips.
// Where a row's bytes live.  ZdDirect: the frame's output in global memory (CG: match sources are read through L2, for
// bytes another SM may have written during the kernel).  ZdWindow (zstd_decode_staged.cu, the chain executor): the recent
// output in a shared-memory window, older bytes in global memory.
template <bool CG>
struct ZdDirect {
	u8* out;
	ZG_DEV u8* dst(u64 pos) const { return out + pos; }
	ZG_DEV void lane_copy(u64 dpos, u64 spos, u32 n) const { zd_lane_copy<CG>(out + dpos, out + spos, n); }
	ZG_DEV void lane_overlap(u64 dpos, u32 off, u32 ml) const { zd_lane_overlap<CG>(out + dpos, off, ml); }
	ZG_DEV void warp_copy(u64 dpos, u64 spos, u32 n) const { zg_warp_copy_t<CG>(out + dpos, out + spos, n); }
	ZG_DEV void warp_match(u64 dpos, u32 off, u32 ml) const { zd_warp_match<CG>(out + dpos, off, ml); }
};

template <class POL>
ZG_DEV u32 zd_exec_row(u64 sq_lane, u32 cnt, const POL& P, u64& o_io, u64 base, u64 cap, const u8* lit, bool lit_rle, u32 rle_byte,
                       u32 regen, u32& lpos_io) {
	u32 lane = zg_lane();
	u64 o = o_io;
	u32 lpos = lpos_io;
	bool act = lane < cnt;
	u64 sq = act ? sq_lane : 0;
	u32 of = (u32)sq & ZD_OFF_MAX, ll = (u32)(sq >> 28) & 0x3ffffu, ml = (u32)(sq >> 46);
	u32 incl = zg_warp_incl_scan(ll + ml), lincl = zg_warp_incl_scan(ll);
	u32 btot = __shfl_sync(ZG_FULL, incl, 31), ltot = __shfl_sync(ZG_FULL, lincl, 31);
	if (lpos + ltot > regen) return ZS_E_CORRUPT;
	if (o + btot > cap) return ZS_E_DST_SMALL;
	u32 rstart = incl - ml;          // my match's start relative to the row's output start
	u64 mstart = o + rstart;         // ... and in the frame output
	if (__any_sync(ZG_FULL, act && (u64)of > mstart - base)) return ZS_E_CORRUPT;
	u8* d = P.dst(mstart - ll);
	u32 lsrc = lpos + (lincl - ll);
	// (a) literals
	u32 longl = __ballot_sync(ZG_FULL, ll > ZD_LANE_COPY_MAX);
	if (ll <= ZD_LANE_COPY_MAX) {
		if (lit_rle) for (u32 k = 0; k < ll; k++) d[k] = (u8)rle_byte;
		else zd_lane_copy<false>(d, lit + lsrc, ll);
	}
	while (longl) {
		int l = __ffs((int)longl) - 1;
		longl &= longl - 1;
		u32 n2 = __shfl_sync(ZG_FULL, ll, l), s2 = __shfl_sync(ZG_FULL, lsrc, l);
		u64 d2 = __shfl_sync(ZG_FULL, (u64)(uintptr_t)d, l);
		if (lit_rle) zg_warp_fill((u8*)(uintptr_t)d2, rle_byte, n2);
		else zg_warp_copy((u8*)(uintptr_t)d2, lit + s2, n2);
	}
	// (b) matches.  need = the lanes below me whose match starts before the end of my source
	//     (rstart grows with the lane: binary search by shuffles; idle lanes sit at the far end)
	i32 rs = act ? (i32)rstart : 0x7fffffff;
	i32 send = (i32)rstart - (i32)of + (i32)zg_min<u32>(ml, of);  // <= 0: the source lies before this row
	u32 nlow = 0;
	ZG_UNROLL
	for (int s = 16; s >= 1; s >>= 1) {
		i32 v = __shfl_sync(ZG_FULL, rs, (int)(nlow + (u32)s - 1u));
		if (v < send) nlow += (u32)s;
	}
	nlow = zg_min<u32>(nlow, lane);
	// ... and of those, not the ones whose match ends at or before my source begins (match ends grow with the
	// lane too): what is left is exactly the lanes whose output my source overlaps.  Waiting for the whole prefix
	// instead would push every later match behind the deepest chain seen so far.
	i32 re = act ? (i32)(rstart + ml) : 0x7fffffff;
	i32 sbeg = (i32)rstart - (i32)of;
	u32 nlo = 0;
	ZG_UNROLL
	for (int s = 16; s >= 1; s >>= 1) {
		i32 v = __shfl_sync(ZG_FULL, re, (int)(nlo + (u32)s - 1u));
		if (v <= sbeg) nlo += (u32)s;
	}
	nlo = zg_min<u32>(nlo, nlow);
	u32 need = ((1u << nlow) - 1u) & ~((1u << nlo) - 1u);
	u32 pending = __ballot_sync(ZG_FULL, act && ml > 0);
	__syncwarp();  // the literals are written
	while (pending) {
		bool ready = ((pending >> lane) & 1u) && !(pending & need);
		bool shortm = ml <= ZD_LANE_COPY_MAX;
		u32 rdy = __ballot_sync(ZG_FULL, ready);
		u32 longm = __ballot_sync(ZG_FULL, ready && !shortm);
		if (ready && shortm) {
			if (of >= ml) P.lane_copy(mstart, mstart - of, ml);
			else P.lane_overlap(mstart, of, ml);
		}
		while (longm) {
			int l = __ffs((int)longm) - 1;
			longm &= longm - 1;
			u32 n2 = __shfl_sync(ZG_FULL, ml, l), o2 = __shfl_sync(ZG_FULL, of, l);
			u64 m2 = __shfl_sync(ZG_FULL, mstart, l);
			if (o2 >= n2) P.warp_copy(m2, m2 - o2, n2);
			else P.warp_match(m2, o2, n2);
		}
		__syncwarp();
		pending &= ~rdy;
	}
	o_io = o + btot;
	lpos_io = lpos + ltot;
	return ZS_OK;
}

// Phase C for the block in flight of the frame viewed by U (uniform): literals, then all sequences.
ZG_DEV void zd_exec_block(ZdWarp* W, ZdLane& U, const u64* seqs, u8* litbuf, ZdHufSave* save) {
	ZdLitHdr h;
	zd_lit_header(U.blk, U.blk_n, h);  // validated in phase A
	const u8* lit;
	bool lit_rle;
	u32 rle_byte;
	u32 r = zd_literals(W, U.flags, U.blk, h, litbuf, save, lit, lit_rle, rle_byte);
	if (r) return zd_fail(U, r);
	u64 o = U.opos;
	u32 lpos = 0;
	u32 lane = zg_lane();
	u64 sq = lane < U.nseq ? seqs[lane] : 0;
	for (u32 s0 = 0; s0 < U.nseq; s0 += 32) {
		u64 sq_next = s0 + 32 + lane < U.nseq ? seqs[s0 + 32 + lane] : 0;  // the next row's records come in while this row executes
		r = zd_exec_row(sq, zg_min<u32>(32u, U.nseq - s0), ZdDirect<false>{U.out}, o, U.base, U.cap, lit, lit_rle, rle_byte, h.regen, lpos);
		if (r) return zd_fail(U, r);
		sq = sq_next;
	}
	// the literals after the last sequence
	u32 rest = h.regen - lpos;
	if (o + rest > U.cap) return zd_fail(U, ZS_E_DST_SMALL);
	if (rest) {
		if (lit_rle) zg_warp_fill(U.out + o, rle_byte, rest);
		else zg_warp_copy(U.out + o, lit + lpos, rest);
		o += rest;
	}
	if (o - U.opos > ZS_BLOCK_MAX) return zd_fail(U, ZS_E_CORRUPT);
	__syncwarp();
	U.opos = o;
	U.nseq = 0;
	if (U.flags & ZD_F_LAST) zd_frame_finish(U);
}


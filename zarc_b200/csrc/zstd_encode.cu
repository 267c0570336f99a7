// K2 + K3: Zstandard block encode.  Replaces the arithmetic of CCtx::compress2 as called at
// crates/zarc/src/encode/lowlevel_frames.rs:30 (libzstd 1.5.5 in the reference).  Compressed bytes
// are not required to equal libzstd's; every block must be valid RFC 8878 that libzstd restores.
//
// Three kernels per chunk of blocks (K2 match -> K3a literals -> K3b sequences), one warp per
// <=128 KiB block pulled from an atomic queue in each.  Splitting by phase keeps every kernel's hot
// code inside the instruction cache (one fused kernel spent 20-35 % of its issue slots waiting for
// instruction fetch) and lets each phase size its own shared memory.  Sequences and literals pass
// between the kernels through a staging area laid out like the chunk's input (a block's sequences
// at 2x, its literals at 1x its offset inside the chunk).
//   K2 match finding: the warp hashes 32 consecutive positions at a time (4-byte hash) against a
//      shared-memory table of 16-bit positions (64 KiB window inside the block), also matching
//      lanes against each other (__match_any_sync) for distances < 32; every lane verifies and
//      extends its own candidate; a warp-uniform greedy+lazy parse picks the matches, resolves
//      repeat-offset codes and gathers literals (histogrammed in shared memory on the way).
//   K3 entropy: length-limited Huffman for literals (tree description FSE-compressed or direct,
//      1 or 4 streams, bit-packing parallel across the warp); FSE for LL/OF/ML codes with
//      Predefined / RLE / FSE_Compressed modes; sequence bitstream written by lane 0.
// Output: the block body in the block's slot of a scratch blob laid out like the input; block
// sizes go to blk_csize (bit 31 = Raw block: body is the input itself).
#include "common.h"
#include "zstd_common.cuh"

#define ZE_WARPS 4
#ifndef ZE_HLOG_MAX
#define ZE_HLOG_MAX 12
#endif
#ifndef ZE_MIN_CTAS
#define ZE_MIN_CTAS 7   // K2: CTAs per SM (shared memory: 7 x (4 x 8064 + 1024 reserved) = 227.5 KiB of the SM's 228)
#endif
// The match finder is bound by the latency of its own dependent steps, so what counts is how many warps an SM holds,
// and that is set by the hash table in shared memory.  The largest table is 63/64 of 2^12 entries: one CTA more per SM
// (28 warps instead of 24) for 1.6 % fewer entries.  Smaller still (-DZE_TAB_FOLD=55u -DZE_MIN_CTAS=8: 32 warps; 48u / 9:
// 36 warps) the kernel keeps getting faster -- 23.7 -> 22.2 -> 21.2 ms per 2 GiB, pack 51.2 -> 53.3 -> 54.8 GB/s -- but
// the ratio pays (C2 level 3: 2.537 -> 2.523 -> 2.512); 63 kept.
#ifndef ZE_TAB_FOLD
#define ZE_TAB_FOLD 63u   // table entries / 64
#endif
#define ZE_TAB_ENTRIES (ZE_TAB_FOLD * 64u)
#ifndef ZE_ENT_CTAS
#define ZE_ENT_CTAS 6   // K3a/K3b: CTAs per SM
#endif
#ifndef ZE_CHUNK_BYTES
#define ZE_CHUNK_BYTES (2ull << 30)  // input bytes per chunk (staging between the kernels = 6x this); 0.25 / 0.5 / 1 / 2 / 4 GiB: 47.0 / 49.8 / 50.1 / 50.8 / 51.0 GB/s pack
#endif
#define ZE_NQ 4  // queue counters per chunk (one per kernel)
#define ZE_MAXSEQ 32768u
#define ZE_MINMATCH 4u
// largest FSE table logs the encoder chooses (the format allows 9 / 9 / 8).  A decoder looks a state up per sequence
// and table; smaller tables of many frames in flight stay cache-resident.
// One below the maxima costs 0.1 % of ratio on the C2 corpus and takes 5 % off the decode kernel.
#ifndef ZE_LL_LOGCAP
#define ZE_LL_LOGCAP (ZS_LL_MAXLOG - 1)
#endif
#ifndef ZE_ML_LOGCAP
#define ZE_ML_LOGCAP (ZS_ML_MAXLOG - 1)
#endif
#ifndef ZE_OF_LOGCAP
#define ZE_OF_LOGCAP (ZS_OF_MAXLOG - 1)
#endif
#ifndef ZE_LANE_CAP
#define ZE_LANE_CAP 64u   // per-lane match extension cap; longer matches are extended by the whole warp
#endif
#define ZE_RAW 0x80000000u

ZG_CONST_TABLE u8 ZS_LL_CODE[64] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 16, 17, 17, 18, 18, 19, 19, 20, 20, 20, 20, 21, 21, 21, 21, 22, 22, 22, 22, 22, 22, 22, 22, 23, 23, 23, 23, 23, 23, 23, 23, 24, 24, 24, 24, 24, 24, 24, 24, 24, 24, 24, 24, 24, 24, 24, 24};
ZG_CONST_TABLE u8 ZS_ML_CODE[128] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 32, 33, 33, 34, 34, 35, 35, 36, 36, 36, 36, 37, 37, 37, 37, 38, 38, 38, 38, 38, 38, 38, 38, 39, 39, 39, 39, 39, 39, 39, 39, 40, 40, 40, 40, 40, 40, 40, 40, 40, 40, 40, 40, 40, 40, 40, 40, 41, 41, 41, 41, 41, 41, 41, 41, 41, 41, 41, 41, 41, 41, 41, 41, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42, 42};

ZG_DEV u32 ze_ll_code(u32 ll) { return ll < 64 ? ZS_LL_CODE[ll] : zs_highbit(ll) + 19; }
ZG_DEV u32 ze_ml_code(u32 mlbase) { return mlbase < 128 ? ZS_ML_CODE[mlbase] : zs_highbit(mlbase) + 36; }

// per-warp global scratch
// seq: offset-or-offBase (17 bits) | litLength << 17 (17 bits) | matchLength << 34
#define ZE_SEQ_OF(q) ((u32)(q) & 0x1ffffu)
#define ZE_SEQ_LL(q) ((u32)((q) >> 17) & 0x1ffffu)
#define ZE_SEQ_ML(q) ((u32)((q) >> 34))
#define ZE_SEQ_PACK(of, ll, ml) ((u64)(of) | ((u64)(ll) << 17) | ((u64)(ml) << 34))
struct ZeBlkMeta {       // per block, handed from kernel to kernel
	u32 nseq;            // ZE_RAW: store the block raw
	u32 nlit;
	u32 litsec;          // size of the literals section K3a wrote (0: give up, store raw)
	u32 logs;            // (K3b, in registers) table logs LL | ML << 8 | OF << 16
	u32 fin[3];          // (K3b, in registers) final states LL, ML, OF (low `log` bits)
	u32 pad;
};
// symbolTT row as the chains read it
struct ZeSymTT {
	u32 dnb;
	i32 dfs;
};

struct ZeEnt {
	u16 hcode[256];       // Huffman code | nbBits << 11
	u8 hweight[256];
	union {               // the Huffman tree build is over before any FSE table exists
		struct {
			u16 sorted_sym[256];
			u32 sorted_cnt[256];
			u32 node_cnt[512];
			u16 node_par[512];
			u8 node_depth[512];
		};
		struct {
			u16 st[3][512];   // FSE state tables: LL, ML, OF (OF also serves the Huffman-weight table)
			ZeSymTT tt[3][64]; // symbolTT rows: deltaNbBits, deltaFindState
			u32 hist3[3][64];
		};
	};
	i16 norm[64];
	u16 cumul[66];
	u8 tsym[512];
	u8 wdesc[192];        // Huffman tree description staging
	u32 window[96];       // bit-packing window (384 B)
};
struct ZeWarp {          // K3a / K3b
	ZeEnt e;
	u32 hist[256];
	u32 misc[16];
};
struct ZeMatchWarp {     // K2
	union {
		u16 htab[ZE_TAB_ENTRIES];
		u32 ring[48];    // repeat-offset assignment, after the parse
	};
};

// ---------------------------------------------------------------------------------------------
// forward bit writer (LSB first), single lane, bounded
struct ZeBitW {
	u8* p;
	u8* end;
	u64 acc;
	u32 nbits;
	bool ovf;
};
ZG_DEV void ze_bw_init(ZeBitW& w, u8* p, u8* end) {
	w.p = p;
	w.end = end;
	w.acc = 0;
	w.nbits = 0;
	w.ovf = false;
}
ZG_DEV_NOINLINE void ze_bw_flush(ZeBitW& w) {
	ZG_UNROLL1
	while (w.nbits >= 8) {
		if (w.p < w.end) *w.p++ = (u8)w.acc;
		else w.ovf = true;
		w.acc >>= 8;
		w.nbits -= 8;
	}
}
ZG_DEV void ze_bw_add(ZeBitW& w, u32 v, u32 nb) {  // nb <= 32
	if (w.nbits + nb > 56) ze_bw_flush(w);
	w.acc |= (u64)(v & (nb >= 32 ? 0xffffffffu : ((1u << nb) - 1u))) << w.nbits;
	w.nbits += nb;
}
// append the end marker and pad; returns one-past-last byte written
ZG_DEV u8* ze_bw_close(ZeBitW& w) {
	ze_bw_add(w, 1, 1);
	ze_bw_flush(w);
	if (w.nbits) {
		if (w.p < w.end) *w.p++ = (u8)w.acc;
		else w.ovf = true;
		w.nbits = 0;
	}
	return w.p;
}

// ---------------------------------------------------------------------------------------------
// FSE compression tables (libzstd's formulation: state table + per-symbol deltaNbBits/deltaFindState)
struct ZeCT {
	u16* st;
	ZeSymTT* tt;
	u32 log;
};
ZG_DEV u32 ze_fse_init_state(const ZeCT& ct, u32 sym) {  // FSE_initCState2: smallest state of sym
	ZeSymTT r = ct.tt[sym];
	u32 nb = (r.dnb + (1u << 15)) >> 16;
	u32 v = (nb << 16) - r.dnb;
	return ct.st[(v >> nb) + r.dfs];
}
ZG_DEV void ze_fse_encode(ZeBitW& w, const ZeCT& ct, u32& state, u32 sym) {
	ZeSymTT r = ct.tt[sym];
	u32 nb = (state + r.dnb) >> 16;
	ze_bw_add(w, state, nb);
	state = ct.st[(state >> nb) + r.dfs];
}
ZG_DEV void ze_fse_flush_state(ZeBitW& w, const ZeCT& ct, u32 state) { ze_bw_add(w, state, ct.log); }

// single lane.  norm may hold -1 ("less than one") entries: only the predefined tables do.
ZG_DEV_NOINLINE void ze_fse_build_ctable(const ZeCT& ct, const i16* norm, u32 maxsym, u8* tsym, u16* cumul) {
	u32 log = ct.log, size = 1u << log;
	u32 high = size - 1;
	cumul[0] = 0;
	ZG_UNROLL1
	for (u32 s = 1; s <= maxsym + 1; s++) {
		i32 n = norm[s - 1];
		if (n == -1) {
			cumul[s] = (u16)(cumul[s - 1] + 1);
			tsym[high--] = (u8)(s - 1);
		} else {
			cumul[s] = (u16)(cumul[s - 1] + n);
		}
	}
	u32 step = (size >> 1) + (size >> 3) + 3, mask = size - 1, pos = 0;
	ZG_UNROLL1
	for (u32 s = 0; s <= maxsym; s++)
		ZG_UNROLL1
		for (i32 i = 0; i < norm[s]; i++) {
			tsym[pos] = (u8)s;
			do {
				pos = (pos + step) & mask;
			} while (pos > high);
		}
	ZG_UNROLL1
	for (u32 u = 0; u < size; u++) {
		u32 s = tsym[u];
		ct.st[cumul[s]++] = (u16)(size + u);
	}
	u32 total = 0;
	ZG_UNROLL1
	for (u32 s = 0; s <= maxsym; s++) {
		i32 n = norm[s];
		if (n == 0) {
			ct.tt[s] = ZeSymTT{((log + 1) << 16) - size, 0};
		} else if (n == 1 || n == -1) {
			ct.tt[s] = ZeSymTT{(log << 16) - size, (i32)total - 1};
			total += 1;
		} else {
			u32 maxbits = log - zs_highbit((u32)n - 1);
			u32 minstate = (u32)n << maxbits;
			ct.tt[s] = ZeSymTT{(maxbits << 16) - minstate, (i32)total - n};
			total += (u32)n;
		}
	}
}
// libzstd's FSE_optimalTableLog
ZG_DEV u32 ze_fse_table_log(u32 maxlog, u32 total, u32 maxsym) {
	u32 maxbits_src = zs_highbit(total - 1) - 2;
	u32 minbits = zg_min<u32>(zs_highbit(total) + 1, zs_highbit(maxsym) + 2);
	u32 log = maxlog;
	if (maxbits_src < log) log = maxbits_src;
	if (minbits > log) log = minbits;
	if (log < 5) log = 5;
	if (log > maxlog) log = maxlog;
	return log;
}
// counts -> normalized counts summing to 2^log, every present symbol >= 1.  Single lane.
ZG_DEV_NOINLINE void ze_fse_normalize(i16* norm, const u32* cnt, u32 total, u32 maxsym, u32 log) {
	u32 size = 1u << log;
	i32 left = (i32)size;
	u32 largest = 0, largest_p = 0;
	ZG_UNROLL1
	for (u32 s = 0; s <= maxsym; s++) {
		u32 c = cnt[s];
		if (c == 0) {
			norm[s] = 0;
			continue;
		}
		u32 scaled = c << log;  // <= 2^15 sequences (or 256 weights) << 9: fits 32 bits
		u32 p = scaled / total;
		u32 rem = scaled - p * total;
		if (p == 0) p = 1;
		else if (p < 8 && rem * 2 > total) p++;  // round small probabilities to nearest
		if (p > largest_p) {
			largest_p = p;
			largest = s;
		}
		norm[s] = (i16)p;
		left -= (i32)p;
	}
	if (left >= 0 || -left < (norm[largest] >> 1)) {
		norm[largest] = (i16)(norm[largest] + left);
		return;
	}
	// rare: too many forced-to-1 symbols.  Take the excess from the largest entries, one at a time.
	ZG_UNROLL1
	while (left < 0) {
		u32 big = 0;
		ZG_UNROLL1
		for (u32 s = 1; s <= maxsym; s++)
			if (norm[s] > norm[big]) big = s;
		norm[big]--;
		left++;
	}
}
// Warp-cooperative versions of the two functions above for the sequence tables (no -1 entries).
// Same results as the single-lane code: libzstd's spread visits slot k of the cumulative order at
// table position (k * step) & mask, and hands out each symbol's states in increasing table position.
ZG_DEV_NOINLINE void ze_fse_build_ctable_warp(const ZeCT& ct, const i16* norm, u32 maxsym, u8* tsym, u16* cumul) {
	u32 lane = zg_lane(), log = ct.log, size = 1u << log;
	u32 s0 = 2 * lane, s1 = s0 + 1;
	u32 n0 = s0 <= maxsym ? (u32)norm[s0] : 0u, n1 = s1 <= maxsym ? (u32)norm[s1] : 0u;
	u32 incl = zg_warp_incl_scan(n0 + n1);
	u32 ex0 = incl - n0 - n1, ex1 = ex0 + n0;
	if (s0 <= maxsym + 1) cumul[s0] = (u16)ex0;
	if (s1 <= maxsym + 1) cumul[s1] = (u16)ex1;
	ZG_UNROLL
	for (int k = 0; k < 2; k++) {
		u32 s = k ? s1 : s0, n = k ? n1 : n0, ex = k ? ex1 : ex0;
		if (s > maxsym) continue;
		if (n == 0) {
			ct.tt[s] = ZeSymTT{((log + 1) << 16) - size, 0};
		} else if (n == 1) {
			ct.tt[s] = ZeSymTT{(log << 16) - size, (i32)ex - 1};
		} else {
			u32 maxbits = log - zs_highbit(n - 1);
			ct.tt[s] = ZeSymTT{(maxbits << 16) - (n << maxbits), (i32)ex - (i32)n};
		}
	}
	__syncwarp();
	u32 step = (size >> 1) + (size >> 3) + 3, mask = size - 1;
	for (u32 k = lane; k < size; k += 32) {
		u32 s = 0;  // the symbol owning slot k: largest s with cumul[s] <= k
		ZG_UNROLL
		for (u32 b = 32; b; b >>= 1) {
			u32 c = s + b;
			if (c <= maxsym && cumul[c] <= k) s = c;
		}
		tsym[(k * step) & mask] = (u8)s;
	}
	__syncwarp();
	for (u32 u0 = 0; u0 < size; u0 += 32) {  // size >= 32
		u32 u = u0 + lane;
		u32 sym = tsym[u];
		u32 peers = __match_any_sync(ZG_FULL, sym);
		u32 rank = (u32)__popc(peers & zg_lanemask_lt());
		u32 base = cumul[sym];
		__syncwarp();
		if (rank == 0) cumul[sym] = (u16)(base + (u32)__popc(peers));
		ct.st[base + rank] = (u16)(size + u);
		__syncwarp();
	}
}
ZG_DEV_NOINLINE void ze_fse_normalize_warp(i16* norm, const u32* cnt, u32 total, u32 maxsym, u32 log) {
	u32 lane = zg_lane();
	u32 size = 1u << log;
	u32 sum = 0, best = 0;
	ZG_UNROLL
	for (int k = 0; k < 2; k++) {
		u32 s = lane + 32 * k;
		u32 c = s <= maxsym ? cnt[s] : 0u;
		u32 p = 0;
		if (c) {
			u32 scaled = c << log;  // <= 2^15 sequences << 9: fits 32 bits
			p = scaled / total;
			u32 rem = scaled - p * total;
			if (p == 0) p = 1;
			else if (p < 8 && rem * 2 > total) p++;
		}
		sum += p;
		best = zg_max<u32>(best, (p << 6) | (63u - s));  // largest p, lowest symbol on ties
		if (s <= maxsym) norm[s] = (i16)p;
	}
	sum = zg_warp_sum(sum);
	best = zg_warp_max(best);
	__syncwarp();
	i32 left = (i32)size - (i32)sum;
	u32 largest = 63u - (best & 63u);
	i32 lp = (i32)(best >> 6);
	if (left >= 0 || -left < (lp >> 1)) {
		if (lane == 0) norm[largest] = (i16)(lp + left);
	} else if (lane == 0) {
		while (left < 0) {  // rare: too many forced-to-1 symbols
			u32 big = 0;
			for (u32 s = 1; s <= maxsym; s++)
				if (norm[s] > norm[big]) big = s;
			norm[big]--;
			left++;
		}
	}
	__syncwarp();
}
// FSE table description (NCount) writer, inverse of zs_read_ncount.  Single lane.  Returns bytes (0 = no room).
ZG_DEV_NOINLINE u32 ze_fse_write_ncount(u8* dst, u32 cap, const i16* norm, u32 maxsym, u32 log) {
	ZeBitW w;
	ze_bw_init(w, dst, dst + cap);
	ze_bw_add(w, log - 5, 4);
	i32 remaining = 1 << log;
	u32 s = 0;
	ZG_UNROLL1
	while (remaining > 0 && s <= maxsym) {
		u32 bits = zs_highbit((u32)remaining + 1) + 1;
		u32 thr = (1u << bits) - 1u - ((u32)remaining + 1u);
		u32 value = (u32)(norm[s] + 1);
		if (value < thr) {
			ze_bw_add(w, value, bits - 1);
		} else {
			u32 v = value < (1u << (bits - 1)) ? value : value + thr;
			ze_bw_add(w, v, bits);
		}
		remaining -= norm[s];
		bool zero = norm[s] == 0;
		s++;
		if (zero) {
			// count the zero symbols that follow, in 2-bit groups (3 = "three more, keep going")
			u32 run = 0;
			ZG_UNROLL1
			while (s + run <= maxsym && norm[s + run] == 0) run++;
			s += run;
			ZG_UNROLL1
			while (run >= 3) {
				ze_bw_add(w, 3, 2);
				run -= 3;
			}
			ze_bw_add(w, run, 2);
		}
	}
	ze_bw_flush(w);
	if (w.nbits) {
		if (w.p < w.end) *w.p++ = (u8)w.acc;
		else w.ovf = true;
	}
	return w.ovf ? 0 : (u32)(w.p - dst);
}

// ---------------------------------------------------------------------------------------------
// Huffman: code lengths (<= 11 bits) from the literal histogram.  Returns maxBits (0 = failure),
// fills e.hweight[0..maxsym], e.hcode[], *maxsym_out.  All lanes call.
ZG_DEV_NOINLINE u32 ze_huf_build(ZeWarp* W, u32* maxsym_out) {
	ZeEnt& e = W->e;
	u32 lane = zg_lane();
	// present symbols, ascending symbol order -> node_cnt/node_par as (cnt, sym) staging
	u32 n = 0;
	ZG_UNROLL1
	for (u32 k = 0; k < 8; k++) {
		u32 s = k * 32 + lane;
		u32 c = W->hist[s];
		u32 b = __ballot_sync(ZG_FULL, c > 0);
		if (c > 0) {
			u32 idx = n + (u32)__popc(b & zg_lanemask_lt());
			e.node_cnt[256 + idx] = c;
			e.node_par[256 + idx] = (u16)s;
		}
		n += (u32)__popc(b);
		e.hweight[s] = 0;
	}
	__syncwarp();
	if (n < 2) return 0;
	u32 maxsym = e.node_par[256 + n - 1];
	// rank sort by (count, symbol)
	ZG_UNROLL1
	for (u32 i = lane; i < n; i += 32) {
		u32 key = (e.node_cnt[256 + i] << 8) | e.node_par[256 + i];
		u32 rank = 0;
		ZG_UNROLL1
		for (u32 j = 0; j < n; j++) rank += ((e.node_cnt[256 + j] << 8) | e.node_par[256 + j]) < key;
		e.sorted_cnt[rank] = key >> 8;
		e.sorted_sym[rank] = (u16)(key & 0xff);
	}
	__syncwarp();
	// The tree.  Only the merge of the two sorted queues is serial (lane 0, the queue heads' counts kept in registers);
	// the leaves' depths (every leaf walks to the root), the weights, their histogram and the canonical codes are
	// lane-parallel.  Same tree, weights and codes as the serial construction.
	u32 total = 0;
	ZG_UNROLL1
	for (u32 i = lane; i < n; i += 32) total += e.sorted_cnt[i];
	total = zg_warp_sum(total);
	const u32 root = 2 * n - 2;
	u32 maxd = 0;
	// (a symbol rarer than total / 2^ZS_HUF_MAXLOG would get a longer code than the format allows: start from the
	// floor that makes such depths unlikely instead of finding it by doubling, one tree build per step)
	ZG_UNROLL1
	for (u32 limit = zg_max<u32>(1u, total >> ZS_HUF_MAXLOG);; limit <<= 1) {
		ZG_UNROLL1
		for (u32 i = lane; i < n; i += 32) e.node_cnt[i] = zg_max<u32>(e.sorted_cnt[i], limit);
		__syncwarp();
		if (lane == 0) {
			u32 q1 = 0, q2 = n, nn = n;
			u32 c1 = e.node_cnt[0], c2 = 0xffffffffu;  // heads of the leaf queue and of the internal-node queue
			ZG_UNROLL1
			while (nn < 2 * n - 1) {
				u32 a, b, ca, cb;
				if (q1 < n && (q2 >= nn || c1 <= c2)) {
					a = q1++;
					ca = c1;
					c1 = q1 < n ? e.node_cnt[q1] : 0xffffffffu;
				} else {
					a = q2++;
					ca = c2;
					c2 = q2 < nn ? e.node_cnt[q2] : 0xffffffffu;
				}
				if (q1 < n && (q2 >= nn || c1 <= c2)) {
					b = q1++;
					cb = c1;
					c1 = q1 < n ? e.node_cnt[q1] : 0xffffffffu;
				} else {
					b = q2++;
					cb = c2;
					c2 = q2 < nn ? e.node_cnt[q2] : 0xffffffffu;
				}
				u32 sum = ca + cb;
				e.node_cnt[nn] = sum;
				if (q2 == nn) c2 = sum;  // the internal queue was empty: the new node is its head
				e.node_par[a] = (u16)nn;
				e.node_par[b] = (u16)nn;
				nn++;
			}
		}
		__syncwarp();
		u32 md = 0;
		ZG_UNROLL1
		for (u32 i = lane; i < n; i += 32) {
			u32 d = 0, k = i;
			ZG_UNROLL1
			while (k != root) {
				k = e.node_par[k];
				d++;
			}
			e.node_depth[i] = (u8)d;
			md = zg_max<u32>(md, d);
		}
		maxd = zg_warp_max(md);
		__syncwarp();
		if (maxd <= ZS_HUF_MAXLOG) break;
	}
	// weights and canonical codes (ascending weight, then ascending symbol: RFC 8878 §4.2.1)
	u32* rk = W->hist;       // [0..12] symbols per weight (the literal histogram has been consumed)
	u32* nx = W->hist + 16;  // [1..12] next code of each weight
	if (lane < 13) rk[lane] = 0;
	__syncwarp();
	ZG_UNROLL1
	for (u32 i = lane; i < n; i += 32) {
		u32 w = maxd + 1 - e.node_depth[i];
		e.hweight[e.sorted_sym[i]] = (u8)w;
		atomicAdd(&rk[w], 1u);
	}
	__syncwarp();
	if (lane == 0) {
		u32 start = 0;
		ZG_UNROLL1
		for (u32 w = 1; w <= maxd; w++) {
			nx[w] = start >> (w - 1);
			start += rk[w] << (w - 1);
		}
		W->misc[0] = maxd;
	}
	__syncwarp();
	ZG_UNROLL1
	for (u32 s0 = 0; s0 <= maxsym; s0 += 32) {
		u32 sy = s0 + lane;
		u32 w = sy <= maxsym ? e.hweight[sy] : 0u;
		u32 peers = __match_any_sync(ZG_FULL, w);
		u32 base = w ? nx[w] : 0u;
		__syncwarp();
		if (w) {
			e.hcode[sy] = (u16)((base + (u32)__popc(peers & zg_lanemask_lt())) | ((maxd + 1 - w) << 11));
			if ((peers & zg_lanemask_lt()) == 0) nx[w] = base + (u32)__popc(peers);
		}
		__syncwarp();
	}
	__syncwarp();
	*maxsym_out = maxsym;
	return W->misc[0];
}

// Huffman tree description into e.wdesc.  Returns its size, 0 if not representable.  All lanes call: the histogram of
// the weights and the FSE table are built by the warp; the FSE stream itself (two interleaved states over <= 255
// weights) is a serial chain and stays with lane 0.
ZG_DEV_NOINLINE u32 ze_huf_write_tree(ZeWarp* W, u32 maxsym) {
	ZeEnt& e = W->e;
	u32 lane = zg_lane();
	u32 nw = maxsym;  // weights 0..maxsym-1 are explicit, the last is implied
	u32 direct = nw <= 128 ? 1 + ((nw + 1) >> 1) : 0;
	u32 fse_size = 0;
	if (nw > 2) {
		u32* cnt = W->hist + 32;  // [13] (scratch: the literal histogram has been consumed)
		if (lane < 13) cnt[lane] = 0;
		__syncwarp();
		ZG_UNROLL1
		for (u32 i = lane; i < nw; i += 32) atomicAdd(&cnt[e.hweight[i]], 1u);
		__syncwarp();
		u32 c = lane < 13 ? cnt[lane] : 0u;
		u32 maxw = 31u - (u32)__clz((int)(__ballot_sync(ZG_FULL, c > 0) | 1u));
		u32 maxc = zg_warp_max(c);
		if (maxc != nw && maxc > 1) {
			u32 log = ze_fse_table_log(6, nw, maxw);
			if (lane == 0) {
				ze_fse_normalize(e.norm, cnt, nw, maxw, log);
				W->misc[2] = ze_fse_write_ncount(e.wdesc + 1, 127, e.norm, maxw, log);
			}
			__syncwarp();
			u32 nc = W->misc[2];
			if (nc) {
				ZeCT ct{e.st[2], e.tt[2], log};
				ze_fse_build_ctable_warp(ct, e.norm, maxw, e.tsym, e.cumul);
				__syncwarp();
				if (lane == 0) {
					// The two-state FSE stream of the weights, serial by nature: kept as short as it can be -- bits gathered
					// in a 64-bit register and handed to shared memory 32 at a time (no per-byte stores, no bounds checks:
					// <= 255 symbols of <= 6 bits fit the 384-byte window); the warp copies the bytes out afterwards.
					u32* win = e.window;
					u64 acc = 0;
					u32 nbits = 0, wi = 0;
					auto put = [&](u32 v, u32 nb) {
						acc |= (u64)(v & ((1u << nb) - 1u)) << nbits;
						nbits += nb;
						if (nbits >= 32) {
							win[wi++] = (u32)acc;
							acc >>= 32;
							nbits -= 32;
						}
					};
					auto enc = [&](u32& state, u32 sym) {
						ZeSymTT r = ct.tt[sym];
						u32 nb = (state + r.dnb) >> 16;
						put(state, nb);
						state = ct.st[(state >> nb) + r.dfs];
					};
					u32 ip = nw, s1, s2;
					// libzstd FSE_compress_usingCTable order: the last two weights seed the two states
					if (nw & 1) {
						s1 = ze_fse_init_state(ct, e.hweight[--ip]);
						s2 = ze_fse_init_state(ct, e.hweight[--ip]);
						enc(s1, e.hweight[--ip]);
					} else {
						s2 = ze_fse_init_state(ct, e.hweight[--ip]);
						s1 = ze_fse_init_state(ct, e.hweight[--ip]);
					}
					ZG_UNROLL1
					while (ip > 0) {
						enc(s2, e.hweight[--ip]);
						enc(s1, e.hweight[--ip]);
					}
					put(s2, log);
					put(s1, log);
					put(1, 1);  // the end marker
					u32 sbytes = 4 * wi + ((nbits + 7) >> 3);
					if (nbits) win[wi] = (u32)acc;
					W->misc[2] = sbytes;
				}
				__syncwarp();
				{
					u32 sbytes = W->misc[2];
					bool fits = nc + sbytes < 128;
					if (fits)
						for (u32 i = lane; i < sbytes; i += 32) e.wdesc[1 + nc + i] = (u8)(e.window[i >> 2] >> (8 * (i & 3)));
					__syncwarp();
					if (lane == 0) W->misc[2] = fits ? 1 + nc + sbytes : 0;
				}
				__syncwarp();
				fse_size = W->misc[2];
			}
			__syncwarp();
		}
	}
	if (fse_size && (direct == 0 || fse_size < direct)) {
		if (lane == 0) e.wdesc[0] = (u8)(fse_size - 1);
		__syncwarp();
		return fse_size;
	}
	if (!direct) return 0;
	if (lane == 0) e.wdesc[0] = (u8)(127 + nw);
	ZG_UNROLL1
	for (u32 i = 2 * lane; i < nw; i += 64) {
		u32 hi = e.hweight[i], lo = i + 1 < nw ? e.hweight[i + 1] : 0;
		e.wdesc[1 + (i >> 1)] = (u8)((hi << 4) | lo);
	}
	__syncwarp();
	return direct;
}

// total code bits of lit[0..m)
ZG_DEV_NOINLINE u32 ze_huf_count_bits(const ZeEnt& e, const u8* lit, u32 m) {
	u32 bits = 0;
	u32 lane = zg_lane();
	u32 b_next = lane < m ? lit[lane] : 0u;  // one trip ahead
	for (u32 i = lane; i < m; i += 32) {
		u32 b = b_next;
		b_next = i + 32 < m ? lit[i + 32] : 0u;
		if (i + 256 < m) zg_prefetch_l1(lit + i + 256);
		bits += e.hcode[b] >> 11;
	}
	return zg_warp_sum(bits);
}

// One Huffman stream for lit[0..m) into dst (exactly `nbytes` bytes, as computed from count_bits).
// The last literal is written first (lowest bits); parallel bit packing through a shared window.
ZG_DEV_NOINLINE void ze_huf_encode_stream(ZeWarp* W, const u8* lit, u32 m, u8* dst, u32 total_bits) {
	ZeEnt& e = W->e;
	u32 lane = zg_lane();
	u32* win = e.window;  // 96 words
	u32 bitpos = 0;       // bits already flushed to dst (multiple of 8) + bits pending in window
	u32 flushed = 0;      // bytes written to dst
	for (u32 i = lane; i < 96; i += 32) win[i] = 0;
	__syncwarp();
	// chunks of 32 lanes x 4 literals, walking from the end of the segment
	for (u32 done = 0; done < m || done == 0; done += 128) {
		// lane handles literals at reverse indices r = done + 4*lane + k  (r = 0 is the last literal)
		if (done + 256 + 4 * lane < m) zg_prefetch_l1(lit + (m - 1 - (done + 256 + 4 * lane)));  // two trips ahead
		u64 acc = 0;
		u32 nb = 0;
		for (u32 k = 0; k < 4; k++) {
			u32 r = done + 4 * lane + k;
			if (r < m) {
				u32 c = e.hcode[lit[m - 1 - r]];
				acc |= (u64)(c & 0x7ff) << nb;
				nb += c >> 11;
			}
		}
		bool is_last = done + 128 >= m;
		u32 incl = zg_warp_incl_scan(nb);
		u32 chunk_bits = __shfl_sync(ZG_FULL, incl, 31);
		u32 start = (bitpos & 7) + incl - nb;  // bit offset inside the window
		if (is_last && lane == 31) {
			// the end marker follows the first literal's code
			acc |= (u64)1 << nb;
			nb += 1;
		}
		if (nb) {
			u32 wi = start >> 5, sh = start & 31;
			u64 lo = acc << sh;
			atomicOr(&win[wi], (u32)lo);
			u32 mid = (u32)(lo >> 32);
			if (mid) atomicOr(&win[wi + 1], mid);
			if (sh) {
				u32 hi = (u32)(acc >> (64 - sh));
				if (hi) atomicOr(&win[wi + 2], hi);
			}
		}
		__syncwarp();
		u32 wbits = (bitpos & 7) + chunk_bits + (is_last ? 1 : 0);
		u32 nbytes = is_last ? (wbits + 7) >> 3 : wbits >> 3;
		for (u32 i = lane; i < nbytes; i += 32) dst[flushed + i] = (u8)(win[i >> 2] >> (8 * (i & 3)));
		__syncwarp();
		// keep the partial byte, clear the rest
		u32 keep = (wbits & 7) && !is_last ? (win[nbytes >> 2] >> (8 * (nbytes & 3))) & 0xff : 0;
		__syncwarp();
		for (u32 i = lane; i < 96; i += 32) win[i] = 0;
		__syncwarp();
		if (lane == 0) win[0] = keep;
		__syncwarp();
		flushed += nbytes;
		bitpos += chunk_bits;
		if (is_last) break;
	}
	(void)total_bits;
}

// ---------------------------------------------------------------------------------------------
// Warp-parallel bit packer: each call, every lane contributes one bit field (<= 96 bits, lane order
// = stream order, low bits first); fields are placed by a warp scan and OR-ed into a shared window
// (96 words), whole bytes are flushed to dst, the partial byte carries over.  All lanes call.
struct ZePack {
	u32* win;
	u8* dst;
	u32 cap;
	u32 flushed;  // bytes written
	u32 pend;     // bits pending in the window (< 8 between calls)
	bool ovf;
};
ZG_DEV void ze_pack_init(ZePack& P, u32* win, u8* dst, u32 cap) {
	P.win = win;
	P.dst = dst;
	P.cap = cap;
	P.flushed = 0;
	P.pend = 0;
	P.ovf = false;
	for (u32 i = zg_lane(); i < 96; i += 32) win[i] = 0;
	__syncwarp();
}
ZG_DEV void ze_pack_chunk(ZePack& P, u64 lo, u32 hi, u32 nb) {
	u32 lane = zg_lane();
	u32 incl = zg_warp_incl_scan(nb);
	u32 chunk_bits = __shfl_sync(ZG_FULL, incl, 31);
	if (nb) {
		u32 start = P.pend + incl - nb;
		u32 wi = start >> 5, sh = start & 31;
		u64 a = lo << sh;
		u32 w0 = (u32)a, w1 = (u32)(a >> 32);
		u32 w2 = sh ? (u32)(lo >> (64 - sh)) : 0;
		u32 w3 = 0;
		if (nb > 64) {  // bits 64.. of the field
			u64 b = (u64)hi << sh;
			w2 |= (u32)b;
			w3 = (u32)(b >> 32);
		}
		if (w0) atomicOr(&P.win[wi], w0);
		if (w1) atomicOr(&P.win[wi + 1], w1);
		if (w2) atomicOr(&P.win[wi + 2], w2);
		if (w3) atomicOr(&P.win[wi + 3], w3);
	}
	__syncwarp();
	u32 total = P.pend + chunk_bits;
	u32 nbytes = total >> 3;
	if (P.flushed + nbytes > P.cap) {
		P.ovf = true;
		nbytes = 0;  // stop writing; the caller discards the block
	}
	for (u32 i = lane; i < nbytes; i += 32) P.dst[P.flushed + i] = (u8)(P.win[i >> 2] >> (8 * (i & 3)));
	u32 keep = (total & 7) ? ((P.win[(total >> 3) >> 2] >> (8 * ((total >> 3) & 3))) & 0xffu) : 0u;
	__syncwarp();
	u32 nwords = (total + 31) >> 5;
	for (u32 i = lane; i <= nwords && i < 96; i += 32) P.win[i] = 0;
	__syncwarp();
	if (lane == 0) P.win[0] = keep;
	__syncwarp();
	P.flushed += nbytes;
	P.pend = total & 7;
}
// flush the last partial byte; returns total bytes
ZG_DEV u32 ze_pack_finish(ZePack& P) {
	if (P.pend) {
		if (P.flushed + 1 > P.cap) P.ovf = true;
		else if (zg_lane() == 0) P.dst[P.flushed] = (u8)P.win[0];
		P.flushed += 1;
		P.pend = 0;
	}
	__syncwarp();
	return P.flushed;
}

// ---------------------------------------------------------------------------------------------
// sequence tables: mode choice (libzstd's heuristic for fast strategies), description, CTable.
// All lanes call.  Writes the description at p (bounded by end).  Returns mode, or 0xff on overflow.
// The predefined tables are built once per CTA (ZePredef); only FSE_Compressed tables are built here.
struct ZePredef {
	u16 st_ll[64], st_ml[64], st_of[32];
	ZeSymTT tt_ll[36], tt_ml[53], tt_of[29];
};
ZG_DEV_NOINLINE u32 ze_seq_table(ZeWarp* W, const ZeCT& predef, u32 t, const u32* cnt, u32 nseq, u32 maxsym, u32 maxlog, u32 defmax, u8*& p,
                                 u8* end, ZeCT& ct) {
	ZeEnt& e = W->e;
	u32 lane = zg_lane();
	u32 c0 = lane <= maxsym ? cnt[lane] : 0u, c1 = lane + 32 <= maxsym ? cnt[lane + 32] : 0u;
	u32 key = zg_warp_max(zg_max<u32>((c0 << 6) | (63u - lane), (c1 << 6) | (31u - lane)));
	u32 most = key >> 6, most_sym = 63u - (key & 63u);
	ct.st = e.st[t];
	ct.tt = e.tt[t];
	if (most == nseq && nseq > 2) {  // RLE_Mode
		if (p >= end) return 0xff;
		if (lane == 0) {
			*p = (u8)most_sym;
			ct.st[0] = 1;                 // a 1-entry table: state never changes, no bits
			ct.tt[most_sym] = ZeSymTT{0u - 1u, -1};  // dnb = (0 << 16) - (1 << 0): no bits; st[(1 >> 0) - 1] = st[0] = 1
		}
		p++;
		ct.log = 0;
		__syncwarp();
		return 1;
	}
	u32 deflog = predef.log;
	u32 dyn_min = ((1u << deflog) * 8) >> 3;
	if (maxsym <= defmax && (nseq < dyn_min || most < (nseq >> (deflog - 1)))) {  // Predefined_Mode
		// copy the CTA's predefined table into this warp's slot: the chains address all three
		// tables of a block uniformly
		for (u32 i = lane; i < (1u << deflog); i += 32) ct.st[i] = predef.st[i];
		for (u32 i = lane; i <= defmax; i += 32) ct.tt[i] = predef.tt[i];
		ct.log = deflog;
		__syncwarp();
		return 0;
	}
	u32 log = ze_fse_table_log(maxlog, nseq, maxsym);
	ze_fse_normalize_warp(e.norm, cnt, nseq, maxsym, log);
	if (lane == 0) W->misc[3] = ze_fse_write_ncount(p, (u32)(end - p), e.norm, maxsym, log);
	__syncwarp();
	u32 nc = W->misc[3];
	__syncwarp();
	if (!nc) return 0xff;
	p += nc;
	ct.log = log;
	ze_fse_build_ctable_warp(ct, e.norm, maxsym, e.tsym, e.cumul);
	return 2;
}

// ---------------------------------------------------------------------------------------------
// K2: match finding over one block.  Returns nseq; *lit_count = literals gathered into S->lit (the
// literals after the last match included).  Sequences land in S->seq with their plain offsets; the
// repeat-offset codes are assigned afterwards by ze_assign_repcodes.
//
// Per window of 32 positions: every lane looks up, verifies and extends its own candidate; a short
// warp-uniform loop only SELECTS the matches (greedy, one-step lazy); everything per sequence --
// literal length, the sequence record, gathering the uncovered bytes into the literal buffer and
// histogramming them -- is then done lane-parallel from the selection mask.
// hlog bits of multiplicative hash; a full-size table (hlog = ZE_HLOG_MAX) is folded onto its ZE_TAB_ENTRIES slots
ZG_DEV u32 ze_hash4(u32 v, u32 hlog) {
	u32 h = (v * 2654435761u) >> (32 - hlog);
	return hlog == ZE_HLOG_MAX ? (h * ZE_TAB_FOLD) >> 6 : h;
}

// set index of a WAYS-way table: (hlog - LW) bits, folded like ze_hash4 when the table is full size
template <u32 LW>
ZG_DEV u32 ze_hash_set(u32 v, u32 hlog) {
	u32 h = (v * 2654435761u) >> (32 - (hlog - LW));
	return hlog == ZE_HLOG_MAX ? (h * ZE_TAB_FOLD) >> 6 : h;
}

// what the level and the --zstd parameters (pack.rs:140-195) resolve to, see ze_resolve_params
struct ZeParams {
	u32 lazy;       // 1: one-step lazy parse (levels >= 3 / strategies greedy and up)
	u32 ways;       // candidates kept per hash set: 1 (levels < 6), 2 (6-8), 4 (>= 9); searchLog
	u32 min_match;  // shortest match emitted (4..7); minMatch
	u32 max_dist;   // largest offset searched (<= 65535: matches never leave the 64 KiB the 16-bit table reaches); windowLog
	u32 hlog_cap;   // hash table log2 (8..12); hashLog
	u32 accel;      // negative levels: -level (1..ZE_ACCEL_MAX); 0 otherwise.  >= 2: strided fast parse (ze_fast_block)
	u32 raw_lit;    // 1: every literals section Raw (negative levels, libzstd's literal compression off)
};
#define ZE_ACCEL_MAX 131072u  // -(the lowest level): the first step is already larger than a block

// 16 bytes at an arbitrary address as four words.  Only aligned words are touched, and words that
// start at or beyond `lim` read as zero (nothing past the block is dereferenced).
ZG_DEV void ze_ld128(const u8* p, const u8* lim, u32 out[4]) {
	uintptr_t a = (uintptr_t)p;
	const u32* w = (const u32*)(a & ~(uintptr_t)3);
	u32 sh = (u32)(a & 3) * 8;
	u32 x[5];
	ZG_UNROLL
	for (int k = 0; k < 5; k++) x[k] = (const u8*)(w + k) < lim ? __ldg(w + k) : 0u;  // (the input is read-only for the whole kernel: global, non-coherent loads)
	ZG_UNROLL
	for (int k = 0; k < 4; k++) out[k] = __funnelshift_r(x[k], x[k + 1], sh);
}
// the same plus the four bytes before p (0 when p is within 4 bytes of the block start `lo`).
// GUARD = false: the caller knows that p + 20 <= lim (no word can start at or beyond lim).
template <bool GUARD>
ZG_DEV u32 ze_ld128_prev(const u8* p, const u8* lo, const u8* lim, u32 out[4]) {
	uintptr_t a = (uintptr_t)p;
	const u32* w = (const u32*)(a & ~(uintptr_t)3);
	u32 sh = (u32)(a & 3) * 8;
	u32 x[5];
	ZG_UNROLL
	for (int k = 0; k < 5; k++) x[k] = (!GUARD || (const u8*)(w + k) < lim) ? __ldg(w + k) : 0u;
	u32 xm = (p >= lo + 4 && (!GUARD || (const u8*)(w - 1) < lim)) ? __ldg(w - 1) : 0u;
	ZG_UNROLL
	for (int k = 0; k < 4; k++) out[k] = __funnelshift_r(x[k], x[k + 1], sh);
	return __funnelshift_r(xm, x[0], sh);
}
// number of leading equal bytes (0..16) of two 16-byte groups
ZG_DEV u32 ze_eq16(const u32 a[4], const u32 b[4]) {
	u32 x0 = a[0] ^ b[0], x1 = a[1] ^ b[1], x2 = a[2] ^ b[2], x3 = a[3] ^ b[3];
	if (x0) return ((u32)__ffs((int)x0) - 1u) >> 3;
	if (x1) return 4u + (((u32)__ffs((int)x1) - 1u) >> 3);
	if (x2) return 8u + (((u32)__ffs((int)x2) - 1u) >> 3);
	if (x3) return 12u + (((u32)__ffs((int)x3) - 1u) >> 3);
	return 16u;
}

// One more candidate for the position `pos` (deeper searches, WAYS > 1): a 4-byte check first, then the same 16 bytes per
// round trip verification as the single-candidate path; kept when longer than what the lane has.
ZG_DEV void ze_try_candidate(const u8* src, const u8* lim, u32 n, u32 pos, i32 cand, u32 v, const u32 own[4], u32 own_before, u32& mlen,
                             u32& moff, u32& bmatch) {
	if (cand < 0) return;
	if (zg_ld32(src + cand) != v) return;
	u32 c[4];
	u32 cand_before = ze_ld128_prev<true>(src + cand, src, lim, c);
	u32 maxl = zg_min<u32>(n - pos, ZE_LANE_CAP);
	u32 l = ze_eq16(own, c);
	while (l < maxl && (l & 15u) == 0) {
		u32 a[4];
		ze_ld128(src + pos + l, lim, a);
		ze_ld128(src + (u32)cand + l, lim, c);
		u32 e = ze_eq16(a, c);
		l += e;
		if (e < 16) break;
	}
	l = zg_min<u32>(l, maxl);
	if (l > mlen) {
		mlen = l;
		moff = pos - (u32)cand;
		bmatch = cand >= 4 ? (u32)__clz((int)(own_before ^ cand_before)) >> 3 : 0u;
	}
}

// A match of L bytes at p (offset O) that the lane-capped extension stopped at ZE_LANE_CAP: the whole warp extends it,
// 128 bytes per step.  Returns the full length.  All lanes call.
ZG_DEV u32 ze_extend_warp(const u8* src, u32 n, u32 p, u32 L, u32 O) {
	u32 lane = zg_lane();
	for (;;) {
		u32 q = p + L + 4 * lane;
		u32 eq = 0;
		if (q + 4 <= n) {
			u32 x = zg_ld32(src + q) ^ zg_ld32(src + q - O);
			eq = x ? (((u32)__ffs((int)x) - 1) >> 3) : 4;
		} else {
			while (q + eq < n && eq < 4 && src[q + eq] == src[q + eq - O]) eq++;
		}
		u32 full = __ballot_sync(ZG_FULL, eq == 4);
		if (full == ZG_FULL) {
			L += 128;
			continue;
		}
		u32 first = (u32)__ffs((int)~full) - 1;
		return L + 4 * first + __shfl_sync(ZG_FULL, eq, (int)first);
	}
}

// WAYS = 1: one 16-bit position per hash (levels < 6).  WAYS = 2 / 4: the table is 2^hlog / WAYS sets of WAYS positions,
// most recent first; every position verifies all of them (and the nearest same-set position of its own window) and keeps
// the longest match -- the deeper search of the higher levels (libzstd: chain searches of 2^searchLog attempts).
template <int WAYS>
ZG_DEV u32 ze_match_block(ZeMatchWarp* W, u64* seq, u8* lit, const u8* src, u32 n, const ZeParams& prm, u32* lit_count) {
	u32 lane = zg_lane();
	u32 ltmask = zg_lanemask_lt();
	const u32 lazy = prm.lazy, minmatch = prm.min_match, maxdist = prm.max_dist;
	constexpr u32 LW = WAYS == 4 ? 2 : WAYS == 2 ? 1 : 0;
	u32 hlog = 8;
	while (hlog < prm.hlog_cap && (1u << hlog) < n) hlog++;
	u16* htab = W->htab;
	const u8* lim = src + n;
	{
		u32* h32 = (u32*)htab;
		for (u32 i = lane; i < zg_min<u32>(1u << hlog, ZE_TAB_ENTRIES) / 2; i += 32) h32[i] = 0;
	}
	__syncwarp();
	u32 mend = 0;      // end of the last match = start of the pending literals
	u32 lpos = 0, nseq = 0, ip = 0;
	while (ip < n && nseq < ZE_MAXSEQ - 32) {
		u32 pos = ip + lane;
		bool inb = pos < n;
		bool valid = pos + 4 <= n;
		zg_prefetch_l2(src + zg_min<u32>(ip + 2048u, n - 1u));
		u32 own[4];
		// away from the block's end (warp-uniform) no load of this window or of its candidates needs a bounds check
		bool inner = ip + 52u <= n;
		u32 own_before = inner ? ze_ld128_prev<false>(src + pos, src, lim, own)
		                       : ze_ld128_prev<true>(src + pos, src, lim, own);  // + the four bytes before this position
		u32 v = own[0];
		u32 mlen = 0, bmatch = 0, moff = 0;
		if (WAYS == 1) {
		u32 h = valid ? ze_hash4(v, hlog) : (0x80000000u | lane);
		u32 te = valid ? htab[h] : 0;
		u32 peers = __match_any_sync(ZG_FULL, h);
		__syncwarp();
		if (valid && (peers >> lane) == 1u) htab[h] = (u16)pos;  // highest lane of each hash group
		// candidate: nearest earlier lane with the same hash, else the table entry
		u32 lower = peers & ltmask;
		i32 cand = -1;
		if (valid && pos >= mend) {
			if (lower) {
				cand = (i32)(ip + (31u - (u32)__clz((int)lower)));
			} else {
				i32 c = (i32)((pos & ~0xffffu) | te);
				if (c >= (i32)pos) c -= 65536;
				cand = c;
			}
			if (cand >= 0 && pos - (u32)cand > maxdist) cand = -1;
		}
		// verify + extend, 16 bytes per memory round trip (both sides loaded before any compare)
		if (cand >= 0) {
			u32 c[4];
			u32 cand_before = inner ? ze_ld128_prev<false>(src + cand, src, lim, c) : ze_ld128_prev<true>(src + cand, src, lim, c);
			if (c[0] == v) {
				u32 maxl = zg_min<u32>(n - pos, ZE_LANE_CAP);
				mlen = ze_eq16(own, c);
				while (mlen < maxl && (mlen & 15u) == 0) {
					u32 a[4];
					ze_ld128(src + pos + mlen, lim, a);
					ze_ld128(src + (u32)cand + mlen, lim, c);
					u32 e = ze_eq16(a, c);
					mlen += e;
					if (e < 16) break;
				}
				mlen = zg_min<u32>(mlen, maxl);
				// equal bytes right before the match, counted down from position pos - 1 (for the catch-up below)
				if (cand >= 4) bmatch = (u32)__clz((int)(own_before ^ cand_before)) >> 3;
			}
		}
		moff = mlen ? pos - (u32)cand : 0;
		} else {
			// ---- set-associative table ----
			u32 set = valid ? ze_hash_set<LW>(v, hlog) : (0x80000000u | lane);
			u64 e = 0;
			if (valid) e = WAYS == 4 ? ((const u64*)htab)[set] : (u64)((const u32*)htab)[set];
			u32 peers = __match_any_sync(ZG_FULL, set);
			__syncwarp();
			if (valid && (peers >> lane) == 1u) {
				// the set's leader (its highest lane) puts the set's positions of this window in front, most recent first
				u64 ne = e;
				u32 m = peers;
				u32 cnt = zg_min<u32>((u32)__popc(m), (u32)WAYS);
				ne = cnt >= (u32)WAYS ? 0ull : ne << (16 * cnt);
				ZG_UNROLL
				for (int k = 0; k < WAYS; k++) {
					if (m) {
						u32 l = 31u - (u32)__clz((int)m);
						m &= ~(1u << l);
						ne |= (u64)((ip + l) & 0xffffu) << (16 * k);
					}
				}
				if (WAYS == 4) ((u64*)htab)[set] = ne;
				else ((u32*)htab)[set] = (u32)ne;
			}
			if (valid && pos >= mend) {
				u32 lower = peers & ltmask;
				if (lower) ze_try_candidate(src, lim, n, pos, (i32)(ip + (31u - (u32)__clz((int)lower))), v, own, own_before, mlen, moff, bmatch);
				ZG_UNROLL
				for (int k = 0; k < WAYS; k++) {
					u32 te = (u32)(e >> (16 * k)) & 0xffffu;
					i32 c = (i32)((pos & ~0xffffu) | te);
					if (c >= (i32)pos) c -= 65536;
					// (an empty slot reads as position 0, like the one-way table: a candidate like any other)
					if (c >= 0 && pos - (u32)c <= maxdist) ze_try_candidate(src, lim, n, pos, c, v, own, own_before, mlen, moff, bmatch);
				}
			}
		}
		__syncwarp();
		// ---- selection ----
		// Greedy with one-step lazy evaluation, resolved without a per-candidate loop: a match is
		// "good" unless the next position holds one that is more than a byte longer (the skipped
		// lane's successor is then itself a candidate, so the first good lane at or after a position
		// is exactly what the serial rule picks); every lane computes where the parse continues if
		// it is taken (first good lane at or after its match end), and the warp only chases that
		// chain from the first good lane.  A selected match is maximal for its offset, so the next
		// one can never be "zero literals + same offset" (ze_assign_repcodes double-checks).
		u32 has = __ballot_sync(ZG_FULL, mlen >= minmatch);
		u32 mlen_up = __shfl_down_sync(ZG_FULL, mlen, 1);
		bool skip = lazy && lane < 31 && mlen >= minmatch && mlen_up > mlen + 1;
		u32 good = has & ~__ballot_sync(ZG_FULL, skip);
		u32 t = lane + mlen;
		u32 nxt = t < 32 ? (u32)__ffs((int)(good & ~((1u << t) - 1u))) - 1u : 0xffffffffu;
		u32 sel = 0;
		u32 cur = mend;
		for (u32 s = (u32)__ffs((int)good) - 1u; s < 32u; s = __shfl_sync(ZG_FULL, nxt, (int)s)) sel |= 1u << s;
		if (sel) {
			u32 i = 31u - (u32)__clz((int)sel);  // only the last selected match can leave the window
			u32 L = __shfl_sync(ZG_FULL, mlen, (int)i), O = __shfl_sync(ZG_FULL, moff, (int)i);
			u32 p = ip + i;
			if (L >= ZE_LANE_CAP && p + L < n) {
				L = ze_extend_warp(src, n, p, L, O);
				if (lane == i) mlen = L;
			}
			cur = p + L;
		}
		// ---- emission (lane-parallel) ----
		u32 below = sel & ltmask;
		u32 my_end = pos + mlen;
		u32 pend = __shfl_sync(ZG_FULL, my_end, below ? (int)(31u - (u32)__clz((int)below)) : 0);
		u32 prev_end = below ? pend : mend;  // end of the nearest match that starts before this position
		bool selme = (sel >> lane) & 1u;
		// a selected match also takes the pending literals right before it that equal the bytes before
		// its source (libzstd's "catch up"), at most 4 and never across the window start: a literal
		// that becomes match length costs no Huffman code
		u32 bext = selme ? zg_min<u32>(bmatch, zg_min<u32>(pos - prev_end, lane)) : 0u;
		u32 my_start = pos - bext;
		u32 above = sel & ~(ltmask | (1u << lane));
		u32 nstart = __shfl_sync(ZG_FULL, my_start, above ? (int)((u32)__ffs((int)above) - 1u) : 0);
		if (selme) seq[nseq + (u32)__popc(below)] = ZE_SEQ_PACK(moff, my_start - prev_end, mlen + bext);
		bool is_lit = inb && !selme && pos >= prev_end && !(above && pos >= nstart);
		u32 lm = __ballot_sync(ZG_FULL, is_lit);
		if (is_lit) lit[lpos + (u32)__popc(lm & ltmask)] = (u8)v;
		lpos += (u32)__popc(lm);
		nseq += (u32)__popc(sel);
		mend = cur;
		ip = zg_max<u32>(ip + 32, cur);
	}
	// the rest (only when the sequence budget ran out)
	{
		u32 start = zg_max<u32>(ip, mend);
		u32 rest = start < n ? n - start : 0;
		for (u32 k = lane; k < rest; k += 32) lit[lpos + k] = src[start + k];
		lpos += rest;
	}
	__syncwarp();
	*lit_count = lpos;
	return nseq;
}

// Levels -2 and below: libzstd's fast-strategy stepping (ZSTD_compressBlock_fast, targetLength = prm.accel) restated
// for a warp.  Positions are probed in pairs (q, q + 1) whose starts are `step` apart: step = accel + 1 right after a
// match and one more for every ZE_STEP_INCR bytes parsed since.  A window is 16 pairs, lane 2k + j probing
// p + k * step + j; only probed positions enter the table (same table, hash and distance limit as ze_match_block).  The
// first probe with a match of min_match bytes or more is taken, extended forward (the lane, then the whole warp) and
// backward as far as the end of the previous match -- a sampled parse lands inside most matches, and without the
// catch-up their heads would stay literals -- then the first probe at or after its end, and so on.  The next window
// starts at the last match's end (or after the window when there was none).  Same outputs as ze_match_block:
// sequences with plain offsets, literals gathered into `lit`.
#define ZE_STEP_INCR 128u
ZG_DEV u32 ze_fast_block(ZeMatchWarp* W, u64* seq, u8* lit, const u8* src, u32 n, const ZeParams& prm, u32* lit_count) {
	u32 lane = zg_lane();
	u32 ltmask = zg_lanemask_lt();
	const u32 minmatch = prm.min_match, maxdist = prm.max_dist;
	u32 hlog = 8;
	while (hlog < prm.hlog_cap && (1u << hlog) < n) hlog++;
	u16* htab = W->htab;
	const u8* lim = src + n;
	{
		u32* h32 = (u32*)htab;
		for (u32 i = lane; i < zg_min<u32>(1u << hlog, ZE_TAB_ENTRIES) / 2; i += 32) h32[i] = 0;
	}
	__syncwarp();
	u32 mend = 0;  // end of the last match = start of the pending literals
	u32 lpos = 0, nseq = 0, ip = 0;
	while (ip < n && nseq < ZE_MAXSEQ - 32) {
		u32 step = prm.accel + 1 + (ip - mend) / ZE_STEP_INCR;  // (<= 2^17 + 2^10: the window's positions fit 32 bits)
		u32 pos = ip + (lane >> 1) * step + (lane & 1);
		bool valid = pos + 4 <= n;
		u32 own[4] = {0, 0, 0, 0};
		if (valid) ze_ld128(src + pos, lim, own);
		u32 v = own[0];
		u32 h = valid ? ze_hash4(v, hlog) : (0x80000000u | lane);
		u32 te = valid ? htab[h] : 0;
		u32 peers = __match_any_sync(ZG_FULL, h);
		// candidate: nearest earlier lane with the same hash, else the table entry
		u32 lower = peers & ltmask;
		u32 lower_pos = __shfl_sync(ZG_FULL, pos, lower ? (int)(31u - (u32)__clz((int)lower)) : (int)lane);
		i32 cand = -1;
		if (valid) {
			if (lower) {
				cand = (i32)lower_pos;
			} else {
				i32 c = (i32)((pos & ~0xffffu) | te);
				if (c >= (i32)pos) c -= 65536;
				cand = c;
			}
			if (cand >= 0 && pos - (u32)cand > maxdist) cand = -1;
		}
		u32 mlen = 0;
		if (cand >= 0) {
			u32 c[4];
			ze_ld128(src + cand, lim, c);
			if (c[0] == v) {
				u32 maxl = zg_min<u32>(n - pos, ZE_LANE_CAP);
				mlen = ze_eq16(own, c);
				while (mlen < maxl && (mlen & 15u) == 0) {
					u32 a[4];
					ze_ld128(src + pos + mlen, lim, a);
					ze_ld128(src + (u32)cand + mlen, lim, c);
					u32 e = ze_eq16(a, c);
					mlen += e;
					if (e < 16) break;
				}
				mlen = zg_min<u32>(mlen, maxl);
			}
		}
		// greedy in position order: the first probe with a match, then the first one at or after its end, and so on
		u32 has = __ballot_sync(ZG_FULL, mlen >= minmatch);
		u32 next = ip + 16 * step;  // where the next window starts: here, or the last match's end
		while (has) {
			u32 i = (u32)__ffs((int)has) - 1u;
			u32 L = __shfl_sync(ZG_FULL, mlen, (int)i), q = __shfl_sync(ZG_FULL, pos, (int)i);
			u32 O = q - (u32)__shfl_sync(ZG_FULL, cand, (int)i);
			if (L >= ZE_LANE_CAP && q + L < n) L = ze_extend_warp(src, n, q, L, O);
			// backward, 32 bytes per step: never before the previous match's end nor before the block
			u32 back = 0;
			for (;;) {
				u32 k = back + lane + 1;
				bool eq = k <= q - mend && k <= q - O && src[q - k] == src[q - O - k];
				u32 all = __ballot_sync(ZG_FULL, eq);
				if (all == ZG_FULL) {
					back += 32;
					continue;
				}
				back += (u32)__ffs((int)~all) - 1u;
				break;
			}
			u32 ll = q - back - mend;
			for (u32 k = lane; k < ll; k += 32) lit[lpos + k] = src[mend + k];
			if (lane == 0) seq[nseq] = ZE_SEQ_PACK(O, ll, L + back);
			lpos += ll;
			nseq++;
			mend = q + L;
			next = mend;
			has &= __ballot_sync(ZG_FULL, pos >= mend);
		}
		// After a match the next window starts at its end with the first step again, as libzstd's parse does.  The probes
		// of this window at or after that point are probed again there, so they stay out of the table (a probe would find
		// itself); the others enter it, the highest lane of each hash group.
		u32 ins = __ballot_sync(ZG_FULL, valid && pos < next);
		if (((ins >> lane) & 1u) && ((peers & ins) >> lane) == 1u) htab[h] = (u16)pos;
		__syncwarp();
		ip = next;
	}
	for (u32 k = lane; k < n - mend; k += 32) lit[lpos + k] = src[mend + k];
	lpos += n - mend;
	__syncwarp();
	*lit_count = lpos;
	return nseq;
}

// Repeat-offset codes (RFC 8878 §3.1.1.5) for all sequences of the block, 32 at a time.
// The decoder's history is a move-to-front list of the three most recently used distinct offsets
// (the parse never emits "zero literals + the offset just used", the one transition that is not
// MTF), so for sequence j: rep0 = the previous sequence's offset, rep1 = the last offset different
// from it (found exactly, by a segmented scan), rep2 = the last one different from both (bounded
// look-back; not finding it only costs a code, the decoder's state is the same either way).
// History slots a block cannot know (blocks after the first are encoded independently) are 0 and
// never match.  Rewrites S->seq[i].of from offset to offBase.  Returns false if the impossible
// transition is met (the caller then stores the block raw).
#define ZE_REP_LOOKBACK 8u
ZG_DEV bool ze_assign_repcodes(ZeMatchWarp* W, u64* seq, u32 nseq, bool first_block) {
	u32 lane = zg_lane();
	u32* ro = W->ring;  // [ZE_REP_LOOKBACK + 32] offsets: the previous chunk's tail, then this chunk
	if (lane < ZE_REP_LOOKBACK) ro[lane] = 0;
	__syncwarp();
	u32 a_carry = 0, b_carry = 0;
	if (first_block) {
		if (lane == 0) {
			ro[ZE_REP_LOOKBACK - 1] = 1;
			ro[ZE_REP_LOOKBACK - 2] = 4;
			ro[ZE_REP_LOOKBACK - 3] = 8;
		}
		a_carry = 1;
		b_carry = 4;
	}
	__syncwarp();
	bool ok = true;
	for (u32 s0 = 0; s0 < nseq; s0 += 32) {
		u32 cnt = zg_min<u32>(32u, nseq - s0);
		bool act = lane < cnt;
		u64 q = act ? seq[s0 + lane] : 0;
		u32 O = ZE_SEQ_OF(q), ll = ZE_SEQ_LL(q);
		u32 olast = __shfl_sync(ZG_FULL, O, (int)cnt - 1);
		if (!act) O = olast;  // idle lanes repeat the last offset: no change points
		ro[ZE_REP_LOOKBACK + lane] = O;
		u32 prevO = __shfl_up_sync(ZG_FULL, O, 1);
		if (lane == 0) prevO = a_carry;
		// rep1 AFTER sequence j: the offset before the last change point at or before j
		i32 chg = (O != prevO) ? (i32)lane : -1;
		for (int d = 1; d < 32; d <<= 1) {
			i32 t = __shfl_up_sync(ZG_FULL, chg, d);
			if ((int)lane >= d) chg = chg > t ? chg : t;
		}
		u32 b_after = __shfl_sync(ZG_FULL, prevO, chg < 0 ? 0 : chg);
		if (chg < 0) b_after = b_carry;
		u32 a = prevO;
		u32 b = __shfl_up_sync(ZG_FULL, b_after, 1);
		if (lane == 0) b = b_carry;
		__syncwarp();
		u32 c = 0;
		for (u32 k = 2; k < 2 + ZE_REP_LOOKBACK - 1; k++) {
			// offsets of sequences j-2, j-3, ... (index ZE_REP_LOOKBACK + lane - k in the ring)
			u32 idx = ZE_REP_LOOKBACK + lane - k;
			if (idx > ZE_REP_LOOKBACK + 31) break;  // (unsigned wrap) beyond the ring
			u32 x = ro[idx];
			if (x == 0) break;
			if (x != a && x != b) {
				c = x;
				break;
			}
		}
		u32 ofb;
		if (ll > 0) {
			if (O == a) ofb = 1;
			else if (O == b) ofb = 2;
			else if (O == c) ofb = 3;
			else ofb = O + 3;
		} else {
			if (O == a) {
				ok = ok && !act;
				ofb = O + 3;
			} else if (O == b) ofb = 1;
			else if (O == c) ofb = 2;
			else if (a > 1 && O == a - 1) ofb = 3;
			else ofb = O + 3;
		}
		if (act) seq[s0 + lane] = ZE_SEQ_PACK(ofb, ll, ZE_SEQ_ML(q));
		a_carry = __shfl_sync(ZG_FULL, O, 31);
		b_carry = __shfl_sync(ZG_FULL, b_after, 31);
		__syncwarp();
		u32 keep = lane < ZE_REP_LOOKBACK ? ro[32 + lane] : 0;
		__syncwarp();
		if (lane < ZE_REP_LOOKBACK) ro[lane] = keep;
		__syncwarp();
	}
	return __all_sync(ZG_FULL, ok);
}

// ---------------------------------------------------------------------------------------------
// A Raw (mode 0) or RLE (mode 1) literals section at p: a header of 1, 2 or 3 bytes (Size_Format by nlit, RFC 8878
// §3.1.1.3.1.1) and the payload.  Returns its end, or null when it does not fit before `end`.  All lanes call.
ZG_DEV u8* ze_literals_plain(const u8* lit, u32 nlit, u32 mode, u8* p, u8* end) {
	u32 lane = zg_lane();
	u32 payload = mode == 1 ? 1 : nlit;
	u32 hdr = nlit < 32 ? 1 : nlit < 4096 ? 2 : 3;
	if (p + hdr + payload > end) return nullptr;
	if (lane == 0) {
		if (hdr == 1) p[0] = (u8)(mode | (nlit << 3));
		else if (hdr == 2) {
			u32 v = mode | (1u << 2) | (nlit << 4);
			p[0] = (u8)v;
			p[1] = (u8)(v >> 8);
		} else {
			u32 v = mode | (3u << 2) | (nlit << 4);
			p[0] = (u8)v;
			p[1] = (u8)(v >> 8);
			p[2] = (u8)(v >> 16);
		}
	}
	p += hdr;
	if (mode == 1) {
		if (lane == 0) p[0] = lit[0];
	} else {
		for (u32 i = lane; i < nlit; i += 32) p[i] = lit[i];
	}
	return p + payload;
}

// K3a: the literals section of one block into dst[0..cap).  Returns its size, or 0 if the block
// cannot end up smaller than raw.  All lanes call.
ZG_DEV u32 ze_literals_section(ZeWarp* W, const u8* lit, u32 nlit, u8* dst, u32 cap) {
	ZeEnt& e = W->e;
	u32 lane = zg_lane();
	if (cap < 16) return 0;
	u8* end = dst + cap;
	u8* p = dst;
	for (u32 i = lane; i < 256; i += 32) W->hist[i] = 0;
	__syncwarp();
	u32 w_next = 4 * lane + 4 <= nlit ? *(const u32*)(lit + 4 * lane) : 0u;  // the next trip's word is on its way during this trip
	for (u32 i0 = 0; i0 < nlit; i0 += 128) {  // 4 literals per lane per trip
		u32 i = i0 + 4 * lane;
		u32 w = w_next;
		w_next = i + 132 <= nlit ? *(const u32*)(lit + i + 128) : 0u;  // the literal buffer of a block is 16-byte aligned
		if (i + 512 < nlit) zg_prefetch_l1(lit + i + 512);
		if (i + 4 <= nlit) {
			atomicAdd(&W->hist[w & 0xff], 1u);
			atomicAdd(&W->hist[(w >> 8) & 0xff], 1u);
			atomicAdd(&W->hist[(w >> 16) & 0xff], 1u);
			atomicAdd(&W->hist[w >> 24], 1u);
		} else {
			for (; i < nlit; i++) atomicAdd(&W->hist[lit[i]], 1u);
		}
	}
	__syncwarp();
	u32 maxc = 0;
	for (u32 k = 0; k < 8; k++) maxc = zg_max<u32>(maxc, W->hist[k * 32 + lane]);
	maxc = zg_warp_max(maxc);
	u32 mode = 0;  // 0 raw, 1 rle, 2 huffman
	u32 maxbits = 0, maxsym = 0, tree = 0;
	u32 sbits[4] = {0, 0, 0, 0}, sbytes[4] = {0, 0, 0, 0};
	u32 streams = nlit < 256 ? 1 : 4;
	u32 seg = (nlit + 3) >> 2;
	u32 comp = 0;
	if (nlit > 1 && maxc == nlit) {
		// (not reached by this library's blocks: every byte value of a block is a literal at least once, so literals of one
		// value come only from a block of one value, and its match finder makes that one literal and one match.  Kept for
		// any caller that hands over such literals; tests/encoder_edge_cases.py asserts no frame has RLE literals.)
		mode = 1;
	} else if (nlit >= 64) {
		maxbits = ze_huf_build(W, &maxsym);
		if (maxbits) {
			tree = ze_huf_write_tree(W, maxsym);
		}
		if (tree) {
			if (streams == 1) {
				sbits[0] = ze_huf_count_bits(e, lit, nlit);
				sbytes[0] = (sbits[0] + 8) >> 3;
				comp = tree + sbytes[0];
			} else {
				for (u32 k = 0; k < 4; k++) {
					u32 m = k < 3 ? seg : nlit - 3 * seg;
					sbits[k] = ze_huf_count_bits(e, lit + k * seg, m);
					sbytes[k] = (sbits[k] + 8) >> 3;
				}
				comp = tree + 6 + sbytes[0] + sbytes[1] + sbytes[2] + sbytes[3];
			}
			if (comp + (nlit >> 6) + 2 < nlit && (streams == 4 || (comp < 1024 && nlit < 1024)) && sbytes[0] < 65536 &&
			    sbytes[1] < 65536 && sbytes[2] < 65536)
				mode = 2;
		}
	}
	if (mode == 2) {
		u32 hdr = (streams == 1 || (comp < 1024 && nlit < 1024)) ? 3 : (comp < 16384 && nlit < 16384) ? 4 : 5;
		if (p + hdr + comp > end) return 0;
		if (lane == 0) {
			if (hdr == 3) {
				u32 v = 2u | ((streams == 1 ? 0u : 1u) << 2) | (nlit << 4) | (comp << 14);
				p[0] = (u8)v;
				p[1] = (u8)(v >> 8);
				p[2] = (u8)(v >> 16);
			} else if (hdr == 4) {
				u32 v = 2u | (2u << 2) | (nlit << 4) | (comp << 18);
				p[0] = (u8)v;
				p[1] = (u8)(v >> 8);
				p[2] = (u8)(v >> 16);
				p[3] = (u8)(v >> 24);
			} else {
				u64 v = 2u | (3u << 2) | ((u64)nlit << 4) | ((u64)comp << 22);
				for (u32 i = 0; i < 5; i++) p[i] = (u8)(v >> (8 * i));
			}
		}
		p += hdr;
		for (u32 i = lane; i < tree; i += 32) p[i] = e.wdesc[i];
		p += tree;
		if (streams == 1) {
			ze_huf_encode_stream(W, lit, nlit, p, sbits[0]);
			p += sbytes[0];
		} else {
			if (lane == 0) {
				p[0] = (u8)sbytes[0];
				p[1] = (u8)(sbytes[0] >> 8);
				p[2] = (u8)sbytes[1];
				p[3] = (u8)(sbytes[1] >> 8);
				p[4] = (u8)sbytes[2];
				p[5] = (u8)(sbytes[2] >> 8);
			}
			p += 6;
			for (u32 k = 0; k < 4; k++) {
				u32 m = k < 3 ? seg : nlit - 3 * seg;
				ze_huf_encode_stream(W, lit + k * seg, m, p, sbits[k]);
				p += sbytes[k];
			}
		}
	} else {
		p = ze_literals_plain(lit, nlit, mode, p, end);
		if (!p) return 0;
	}
	__syncwarp();
	__syncwarp();
	return (u32)(p - dst);
}

// K3a of the negative levels: a Raw literals section, the header and a copy.  Same contract as ze_literals_section.
ZG_DEV u32 ze_literals_raw(const u8* lit, u32 nlit, u8* dst, u32 cap) {
	if (cap < 16) return 0;
	u8* p = ze_literals_plain(lit, nlit, 0, dst, dst + cap);
	__syncwarp();
	return p ? (u32)(p - dst) : 0u;
}

// K3b1: sequence codes + histograms, table modes, table descriptions into dst[0..cap) (dst = just
// after the literals section), compression tables into the table arena.  Returns the bytes written
// (header + descriptions), 0 when it does not fit.  All lanes call.
ZG_DEV u32 ze_sequences_tables(ZeWarp* W, ZePredef* P, const u64* seq, u32* codes, u32 nseq, u8* dst, u32 cap, ZeBlkMeta& M) {
	ZeEnt& e = W->e;
	u32 lane = zg_lane();
	u8* end = dst + cap;
	u8* p = dst;
	if (p + 4 > end) return 0;
	if (nseq == 0) {
		if (lane == 0) *p = 0;
		return 1;
	}
	if (lane == 0) {
		if (nseq < 128) p[0] = (u8)nseq;
		else if (nseq < 0x7F00) {
			p[0] = (u8)((nseq >> 8) + 128);
			p[1] = (u8)nseq;
		} else {
			p[0] = 255;
			p[1] = (u8)(nseq - 0x7F00);
			p[2] = (u8)((nseq - 0x7F00) >> 8);
		}
	}
	p += nseq < 128 ? 1 : nseq < 0x7F00 ? 2 : 3;
	// codes + histograms
	for (u32 i = lane; i < 3 * 64; i += 32) (&e.hist3[0][0])[i] = 0;
	__syncwarp();
	u32 mx_ll = 0, mx_ml = 0, mx_of = 0;
	u64 q_next = lane < nseq ? seq[lane] : 0;  // the records of the next trip are on their way while this one is coded
	for (u32 i = lane; i < nseq; i += 32) {
		u64 q = q_next;
		q_next = i + 32 < nseq ? seq[i + 32] : 0;
		if (i + 128 < nseq) zg_prefetch_l1(seq + i + 128);
		u32 lc = ze_ll_code(ZE_SEQ_LL(q)), mc = ze_ml_code(ZE_SEQ_ML(q) - 3), oc = zs_highbit(ZE_SEQ_OF(q));
		codes[i] = lc | (mc << 8) | (oc << 16);
		atomicAdd(&e.hist3[0][lc], 1u);
		atomicAdd(&e.hist3[1][mc], 1u);
		atomicAdd(&e.hist3[2][oc], 1u);
		mx_ll = zg_max<u32>(mx_ll, lc);
		mx_ml = zg_max<u32>(mx_ml, mc);
		mx_of = zg_max<u32>(mx_of, oc);
	}
	mx_ll = zg_warp_max(mx_ll);
	mx_ml = zg_warp_max(mx_ml);
	mx_of = zg_warp_max(mx_of);
	__syncwarp();
	ZeCT ct3[3];  // LL, ML, OF
	{
		u8* q = p + 1;  // after the modes byte
		ZeCT pd_ll{P->st_ll, P->tt_ll, 6}, pd_ml{P->st_ml, P->tt_ml, 6}, pd_of{P->st_of, P->tt_of, 5};
		u32 m_ll = ze_seq_table(W, pd_ll, 0, e.hist3[0], nseq, mx_ll, ZE_LL_LOGCAP, 35, q, end, ct3[0]);
		if (m_ll == 0xff) return 0;
		u32 m_of = ze_seq_table(W, pd_of, 2, e.hist3[2], nseq, mx_of, ZE_OF_LOGCAP, 28, q, end, ct3[2]);
		if (m_of == 0xff) return 0;
		u32 m_ml = ze_seq_table(W, pd_ml, 1, e.hist3[1], nseq, mx_ml, ZE_ML_LOGCAP, 52, q, end, ct3[1]);
		if (m_ml == 0xff) return 0;
		if (lane == 0) *p = (u8)((m_ll << 6) | (m_of << 4) | (m_ml << 2));
		p = q;
	}
	M.logs = ct3[0].log | (ct3[1].log << 8) | (ct3[2].log << 16);
	__syncwarp();
	return (u32)(p - dst);
}

// The three FSE state chains of one block (last sequence first, libzstd's ZSTD_encodeSequences order), leaving
// per sequence the bits each chain emits as a 16-bit field (value | nbBits << 12) of a 64-bit word:
// LL | ML << 16 | OF << 32.
// A chain is serial -- the state after a step depends on the state before it -- but it forgets: encoding a symbol
// of normalized count c keeps only which of c sub-ranges the old state was in, so two walks over the same symbols
// from different states merge after a few steps and stay merged; across a symbol of count 1 (a single state:
// nbBits = tableLog, (state >> tableLog) == 1, next state st[1 + deltaFindState]) they merge at once.  So each
// chain is cut into ZE_CHAIN_LANES ranges of steps, one lane each.  A lane looks upwards from its range for the
// nearest count-1 symbol (or the chain's start) within ZE_CHAIN_WARM steps; from there the state is exact.
// Failing that it starts ZE_CHAIN_WARM steps up from a guessed state.  It walks down to its range without output
// and then produces its range.  Afterwards the ranges are checked in chain order: a lane that started from a guess
// must have entered its range in the state the lane above left off in; if not (rare) it walks its range again
// from the right state.  The fields are bit for bit those of the serial walk.  All lanes call; fills M.fin.
#define ZE_CHAIN_LANES 10u
#ifndef ZE_CHAIN_AHEAD
#define ZE_CHAIN_AHEAD 4     // steps whose codes and table rows are fetched before the serial state look-ups of a trip
#endif
#ifndef ZE_CHAIN_WARM
#define ZE_CHAIN_WARM 160u  // (sweep on the C2 corpus: 48 / 64 / 96 / 128 / 160 / 192 / 256 steps -> 5.08 / 4.77 / 4.40 / 4.24 / 4.19 / 4.20 / 4.27 ms per GB)
#endif
struct ZeChainRun {
	const u32* codes;
	const u16* st;
	const ZeSymTT* tt;
	u16* out;
	u32 sh;
};
// steps from-1 .. to (descending) from `state`; ZE_CHAIN_AHEAD per trip, the codes and their table rows fetched up front so
// that only the state look-ups are serial
ZG_DEV u32 ze_chain_walk(const ZeChainRun& R, u32 state, u32 from, u32 to, bool emit) {
	u32 i = from;
	ZG_UNROLL1
	while (i > to) {
		zg_prefetch_l1(R.codes + (i > 48u ? i - 48u : 0u));  // the walk runs down the codes: the sector a dozen trips on
		u32 m = zg_min<u32>((u32)ZE_CHAIN_AHEAD, i - to);
		ZeSymTT r[ZE_CHAIN_AHEAD];
		ZG_UNROLL
		for (u32 k = 0; k < ZE_CHAIN_AHEAD; k++)
			if (k < m) r[k] = R.tt[(R.codes[i - 1 - k] >> R.sh) & 0xff];
		ZG_UNROLL
		for (u32 k = 0; k < ZE_CHAIN_AHEAD; k++) {
			if (k < m) {
				u32 nb = (state + r[k].dnb) >> 16;
				if (emit) R.out[4 * (i - 1 - k)] = (u16)((state & ((1u << nb) - 1u)) | (nb << 12));
				state = R.st[(state >> nb) + r[k].dfs];
			}
		}
		i -= m;
	}
	return state;
}
ZG_DEV void ze_sequences_chains(ZeWarp* W, const u32* codes, u16* stb16, ZeBlkMeta& M) {
	ZeEnt& e = W->e;
	u32 lane = zg_lane();
	u32 nseq = M.nseq;
	u32 S = nseq - 1;  // steps: step j encodes codes[j], j = S-1 .. 0; the chain starts from codes[nseq - 1]
	u32 t = lane / ZE_CHAIN_LANES, sub = lane % ZE_CHAIN_LANES;
	u32* xch = W->hist;  // per lane: state on entering the range | state on leaving it << 16 (the literal histogram is not in use here)
	bool live = false, exact = true;
	u32 hi = 0, lo = 0, s_in = 0, s_out = 0, log = 0;
	ZeChainRun R{codes, nullptr, nullptr, nullptr, 0};
	if (t < 3) {
		R.sh = 8 * t;  // codes = ll | ml << 8 | of << 16; table index 0 LL, 1 ML, 2 OF
		R.st = e.st[t];
		R.tt = e.tt[t];
		R.out = stb16 + t;  // stride 4
		log = (M.logs >> R.sh) & 0xff;
		u32 reset_dnb = (log << 16) - (1u << log);  // deltaNbBits of a symbol with a single state
		u32 len = (S + ZE_CHAIN_LANES - 1) / ZE_CHAIN_LANES;
		hi = S - zg_min<u32>(S, sub * len);
		lo = S - zg_min<u32>(S, (sub + 1) * len);
		if (sub == 0) R.out[4 * S] = 0;
		live = hi > lo || (sub == 0 && S == 0);
		if (live) {
			ZeCT ct{e.st[t], e.tt[t], log};
			u32 top = zg_min<u32>(S, hi + ZE_CHAIN_WARM);
			u32 from = hi, state = 0;
			bool found = false;
			ZG_UNROLL1
			while (from < top) {
				ZeSymTT r = R.tt[(codes[from] >> R.sh) & 0xff];
				if (r.dnb == reset_dnb) {
					state = R.st[1 + r.dfs];
					found = true;
					break;
				}
				from++;
			}
			if (!found) {
				// the chain's start if it is within reach, else a guess: walk as if the chain started at `top`
				state = ze_fse_init_state(ct, (codes[top] >> R.sh) & 0xff);
				from = top;
				exact = top == S;
			}
			s_in = ze_chain_walk(R, state, from, hi, false);
			s_out = ze_chain_walk(R, s_in, hi, lo, true);
			xch[lane] = s_in | (s_out << 16);
		}
	}
	__syncwarp();
	// in chain order: a guessed start must have merged with the true chain before the range began
	ZG_UNROLL1
	for (u32 k = 1; k < ZE_CHAIN_LANES; k++) {
		bool redo = false;
		u32 s_true = 0;
		if (live && sub == k && !exact) {
			s_true = xch[lane - 1] >> 16;  // the lane above holds the range above (its final state, corrected if need be)
			redo = s_true != s_in;
		}
		if (__any_sync(ZG_FULL, redo)) {
			if (redo) {
				s_out = ze_chain_walk(R, s_true, hi, lo, true);
				xch[lane] = s_true | (s_out << 16);
			}
		}
		__syncwarp();
	}
	if (live && lo == 0) W->misc[8 + t] = s_out & ((1u << log) - 1u);
	__syncwarp();
	M.fin[0] = W->misc[8];
	M.fin[1] = W->misc[9];
	M.fin[2] = W->misc[10];
	__syncwarp();
}

// K3b3: the sequence bitstream of one block into dst[0..cap).  Every lane assembles one sequence's
// bit field (<= 89 bits: OF,ML,LL state bits then LL,ML,OF extra bits), a warp scan places it, and
// the fields are OR-ed into a shared window.  Returns the bytes written, 0 when it does not fit.
ZG_DEV u32 ze_sequences_pack(ZeWarp* W, const u64* seq, const u32* codes, const u64* stb, const ZeBlkMeta& M, u8* dst, u32 cap) {
	ZeEnt& e = W->e;
	u32 lane = zg_lane();
	u32 nseq = M.nseq;
	u32 logs[3] = {M.logs & 0xff, (M.logs >> 8) & 0xff, M.logs >> 16};
	ZePack pk;
	ze_pack_init(pk, e.window, dst, cap);
	// (the three loads of the next trip are issued before this trip's fields are assembled and packed)
	u32 c_next = 0;
	u64 sb_next = 0, q_next = 0;
	if (lane < nseq) {
		u32 i = nseq - 1 - lane;
		c_next = codes[i];
		sb_next = stb[i];
		q_next = seq[i];
	}
	for (u32 hi = nseq; hi > 0; hi -= zg_min<u32>(hi, 32u)) {
		u64 lo64 = 0;
		u32 hi32 = 0, nb = 0;
		u32 c = c_next;
		u64 sb = sb_next, q = q_next;
		if (hi > 32 && lane < hi - 32) {
			u32 i = hi - 33 - lane;
			c_next = codes[i];
			sb_next = stb[i];
			q_next = seq[i];
			if (i >= 96) {  // and the lines three trips further down are asked into L1
				zg_prefetch_l1(stb + i - 96);
				zg_prefetch_l1(seq + i - 96);
			}
		}
		if (lane < hi) {
			u32 lc = c & 0xff, mc = (c >> 8) & 0xff, oc = c >> 16;
			u32 a = (u32)(sb >> 32) & 0xffff, b = (u32)(sb >> 16) & 0xffff, d = (u32)sb & 0xffff;
			lo64 = a & 0xfff;
			nb = a >> 12;
			lo64 |= (u64)(b & 0xfff) << nb;
			nb += b >> 12;
			lo64 |= (u64)(d & 0xfff) << nb;
			nb += d >> 12;
			lo64 |= (u64)(ZE_SEQ_LL(q) - ZS_LL_BASE[lc]) << nb;
			nb += ZS_LL_BITS[lc];
			lo64 |= (u64)(ZE_SEQ_ML(q) - ZS_ML_BASE[mc]) << nb;
			nb += ZS_ML_BITS[mc];  // <= 58 bits so far
			u64 ox = ZE_SEQ_OF(q) - (1u << oc);
			lo64 |= ox << nb;
			if (nb + oc > 64) hi32 = (u32)(ox >> (64 - nb));
			nb += oc;
		}
		ze_pack_chunk(pk, lo64, hi32, nb);
	}
	{
		// final states ML, OF, LL then the end marker (lane 0 only contributes)
		u64 lo64 = 0;
		u32 nb = 0;
		if (lane == 0) {
			lo64 = M.fin[1];
			nb = logs[1];
			lo64 |= (u64)M.fin[2] << nb;
			nb += logs[2];
			lo64 |= (u64)M.fin[0] << nb;
			nb += logs[0];
			lo64 |= (u64)1 << nb;
			nb += 1;
		}
		ze_pack_chunk(pk, lo64, 0, nb);
	}
	u32 bytes = ze_pack_finish(pk);
	__syncwarp();
	return pk.ovf ? 0 : bytes;
}

struct ZeBlk {
	u32 f;         // file
	u32 n;         // block bytes
	u64 j;         // block index inside the file
	u64 soff;      // offset of the block in the staging blob
};
// everything the three kernels need to find a block and its staging
struct ZeJob {
	const u8* blob;
	const u64* file_off;
	const u64* comp_off;
	const u64* file_len;
	const u32* ulist;
	const u64* blk_base;
	u32 nuniq;
	u64 nblocks;
	u8* comp;          // encoded-block staging blob, laid out like the unique inputs
	u32* blk_csize;
	ZeBlkMeta* meta;   // [nblocks]
	u64* seqbuf;       // chunk staging: sequences (8 B per 4 input bytes)
	u8* litbuf;        // chunk staging: literals (1 B per input byte)
	u32* codebuf;      // chunk staging: sequence codes (4 B per 4 input bytes)
	u64* stbbuf;       // chunk staging: FSE state bits (8 B per 4 input bytes)
	const u64* bounds; // [nchunks + 1] first block of every chunk
	const u32* order;  // [nblocks] hand-out order: the blocks of each chunk, largest first (or null: index order)
	const struct ZeBlk* info;  // [nblocks] block -> (file, size, index, staging offset), or null: binary search (ze_locate)
	u64 chunk_bytes;
};
// block -> (unique file, block index): last u with blk_base[u] <= b
ZG_DEV ZeBlk ze_locate(const ZeJob& J, u64 b) {
	u32 lo = 0, hi = J.nuniq - 1;
	while (lo < hi) {
		u32 mid = (lo + hi + 1) >> 1;
		if (J.blk_base[mid] <= b) lo = mid;
		else hi = mid - 1;
	}
	ZeBlk B;
	B.f = J.ulist[lo];
	B.j = b - J.blk_base[lo];
	u64 flen = J.file_len[B.f];
	u64 boff = B.j * ZS_BLOCK_MAX;
	B.n = (u32)zg_min<u64>(ZS_BLOCK_MAX, flen - zg_min<u64>(flen, boff));
	B.soff = J.comp_off[B.f] + boff;
	return B;
}
// the same from the table k_ze_order_scatter filled (one load instead of a 20-step search per block and kernel)
ZG_DEV ZeBlk ze_block(const ZeJob& J, u64 b) { return J.info ? J.info[b] : ze_locate(J, b); }
// next block of chunk k from the kernel's queue; false when the chunk is exhausted
ZG_DEV bool ze_next_block(const ZeJob& J, u32 chunk, u32* queue, u64& b) {
	u32 t = 0;
	if (zg_lane() == 0) t = atomicAdd(queue, 1u);
	t = __shfl_sync(ZG_FULL, t, 0);
	b = J.bounds[chunk] + t;
	if (b >= J.bounds[chunk + 1]) return false;
	if (J.order) b = J.order[b];
	return true;
}

// first block of every chunk: chunk k holds the blocks whose staging offset is in [k, k+1) * chunk_bytes
__global__ void __launch_bounds__(128) k_ze_chunk_bounds(ZeJob J, u32 nchunks, u64* bounds) {
	u32 k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k > nchunks) return;
	if (k == nchunks) {
		bounds[k] = J.nblocks;
		return;
	}
	u64 want = (u64)k * J.chunk_bytes;
	u64 lo = 0, hi = J.nblocks;  // first block with soff >= want
	while (lo < hi) {
		u64 mid = (lo + hi) >> 1;
		if (ze_locate(J, mid).soff >= want) hi = mid;
		else lo = mid + 1;
	}
	bounds[k] = lo;
}

// Hand-out order.  The queues give out blocks one at a time, and a warp needs milliseconds for a full
// 128 KiB block but microseconds for a 1 KiB file: in index order each kernel would end with a tail as
// long as its biggest block.  So the blocks of every chunk are handed out largest first (counting sort
// by size, ZE_OBINS bins per chunk; the order inside a bin does not matter).
#define ZE_OBINS 256u
ZG_DEV u32 ze_obin(u32 n) { return ZE_OBINS - 1u - zg_min<u32>(n >> 9, ZE_OBINS - 1u); }
ZG_DEV size_t ze_obin_slot(const ZeJob& J, const ZeBlk& B, u32 nchunks) {
	return (size_t)zg_min<u64>(B.soff / J.chunk_bytes, nchunks - 1u) * ZE_OBINS + ze_obin(B.n);  // same chunk as k_ze_chunk_bounds
}
__global__ void __launch_bounds__(256) k_ze_order_count(ZeJob J, u32 nchunks, u32* bins) {
	u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (b >= J.nblocks) return;
	atomicAdd(&bins[ze_obin_slot(J, ze_locate(J, b), nchunks)], 1u);
}
// one warp per chunk: exclusive scan of its bins, starting at the chunk's first block
__global__ void __launch_bounds__(32) k_ze_order_scan(ZeJob J, u32* bins) {
	u32* c = bins + (size_t)blockIdx.x * ZE_OBINS;
	u32 lane = threadIdx.x;
	u32 run = (u32)J.bounds[blockIdx.x];
	for (u32 k0 = 0; k0 < ZE_OBINS; k0 += 32) {
		u32 v = c[k0 + lane];
		u32 incl = zg_warp_incl_scan(v);
		c[k0 + lane] = run + incl - v;
		run += __shfl_sync(ZG_FULL, incl, 31);
	}
}
__global__ void __launch_bounds__(256) k_ze_order_scatter(ZeJob J, u32 nchunks, u32* bins, u32* order, ZeBlk* info) {
	u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (b >= J.nblocks) return;
	ZeBlk B = ze_locate(J, b);
	info[b] = B;
	order[atomicAdd(&bins[ze_obin_slot(J, B, nchunks)], 1u)] = (u32)b;
}

// K2.  WAYS = 0: the strided fast parse of levels -2 and below
template <int WAYS>
__global__ void __launch_bounds__(ZE_WARPS * 32, ZE_MIN_CTAS) k_zstd_match_blocks(ZeJob J, u32 chunk, u32* queue, ZeParams prm) {
	ZG_DYN_SMEM(ZeMatchWarp, sm);
	ZeMatchWarp* W = &sm[threadIdx.x >> 5];
	u32 lane = threadIdx.x & 31;
	u64 b;
	while (ze_next_block(J, chunk, queue, b)) {
		ZeBlk B = ze_block(J, b);
		u64 rel = B.soff - (u64)chunk * J.chunk_bytes;
		u64* seq = J.seqbuf + (rel >> 2);
		u8* lit = J.litbuf + rel;
		u32 nseq = ZE_RAW, nlit = 0;
		if (B.n >= 16) {
			const u8* src = J.blob + J.file_off[B.f] + B.j * ZS_BLOCK_MAX;
			if constexpr (WAYS == 0) nseq = ze_fast_block(W, seq, lit, src, B.n, prm, &nlit);
			else nseq = ze_match_block<WAYS>(W, seq, lit, src, B.n, prm, &nlit);
			__syncwarp();
			// later blocks of a frame are encoded independently of their predecessors: unknown history
			if (!ze_assign_repcodes(W, seq, nseq, B.j == 0)) nseq = ZE_RAW;
		}
		__syncwarp();
		if (lane == 0) {
			J.meta[b].nseq = nseq;
			J.meta[b].nlit = nlit;
		}
	}
}

// K3a.  raw_lit: Raw sections only (negative levels): no histogram, no Huffman
__global__ void __launch_bounds__(ZE_WARPS * 32, ZE_ENT_CTAS) k_zstd_literals(ZeJob J, u32 chunk, u32* queue, u32 raw_lit) {
	ZG_DYN_SMEM(ZeWarp, sm);
	ZeWarp* W = &sm[threadIdx.x >> 5];
	u32 lane = threadIdx.x & 31;
	u64 b;
	while (ze_next_block(J, chunk, queue, b)) {
		ZeBlkMeta m = J.meta[b];
		u32 litsec = 0;
		if (m.nseq != ZE_RAW) {
			ZeBlk B = ze_block(J, b);
			u64 rel = B.soff - (u64)chunk * J.chunk_bytes;
			litsec = raw_lit ? ze_literals_raw(J.litbuf + rel, m.nlit, J.comp + B.soff, B.n - 1)
			                 : ze_literals_section(W, J.litbuf + rel, m.nlit, J.comp + B.soff, B.n - 1);
		}
		__syncwarp();
		if (lane == 0) J.meta[b].litsec = litsec;
	}
}

// K3b
__global__ void __launch_bounds__(ZE_WARPS * 32, ZE_ENT_CTAS) k_zstd_sequences(ZeJob J, u32 chunk, u32* queue) {
	ZG_DYN_SMEM(ZeWarp, sm);
	u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	ZeWarp* W = &sm[warp];
	ZePredef* P = (ZePredef*)(sm + ZE_WARPS);
	if (threadIdx.x == 0) {  // the predefined compression tables, once per (persistent) CTA
		ZeEnt& e = W->e;
		ze_fse_build_ctable(ZeCT{P->st_ll, P->tt_ll, 6}, ZS_LL_DEFAULT_NORM, 35, e.tsym, e.cumul);
		ze_fse_build_ctable(ZeCT{P->st_ml, P->tt_ml, 6}, ZS_ML_DEFAULT_NORM, 52, e.tsym, e.cumul);
		ze_fse_build_ctable(ZeCT{P->st_of, P->tt_of, 5}, ZS_OF_DEFAULT_NORM, 28, e.tsym, e.cumul);
	}
	__syncthreads();
	u64 b;
	while (ze_next_block(J, chunk, queue, b)) {
		ZeBlkMeta m = J.meta[b];
		ZeBlk B = ze_block(J, b);
		u32 csize = 0;
		if (m.nseq != ZE_RAW && m.litsec) {
			u64 rel = B.soff - (u64)chunk * J.chunk_bytes;
			const u64* seq = J.seqbuf + (rel >> 2);
			u32* codes = J.codebuf + (rel >> 2);
			u64* stb = J.stbbuf + (rel >> 2);
			u8* dst = J.comp + B.soff + m.litsec;
			u32 cap = B.n - 1 - m.litsec;
			u32 hdr = ze_sequences_tables(W, P, seq, codes, m.nseq, dst, cap, m);
			if (hdr && m.nseq == 0) {
				csize = m.litsec + hdr;
			} else if (hdr) {
				__syncwarp();
				ze_sequences_chains(W, codes, (u16*)stb, m);
				u32 sz = ze_sequences_pack(W, seq, codes, stb, m, dst + hdr, cap - hdr);
				if (sz) csize = m.litsec + hdr + sz;
			}
		}
		__syncwarp();
		if (lane == 0) J.blk_csize[b] = csize ? csize : (ZE_RAW | B.n);
	}
}

// input bytes per chunk; tests shrink it to exercise the multi-chunk path (multiple of 16)
static u64 g_ze_chunk_bytes = ZE_CHUNK_BYTES;
extern "C" void zg_internal_set_encode_chunk_bytes(u64 v) { g_ze_chunk_bytes = v ? (v + 15) & ~(u64)15 : ZE_CHUNK_BYTES; }

// The compression level and the advanced parameters of the CLI's --zstd option (pack.rs:140-195; libzstd's
// ZSTD_cParameter numbers) as this match finder honours them.  Level -> strategy follows libzstd's table in spirit:
// levels 1-2 (fast, dfast) parse greedily, 3-5 add one-step lazy evaluation, 6-8 search two candidates per position,
// 9 and up four.  An explicit strategy / searchLog / hashLog / minMatch / windowLog overrides what the level implies:
//   strategy   1-2 greedy, 3-5 lazy, 6-9 lazy + 4 candidates          searchLog  candidates = 2^min(searchLog, 2)
//   hashLog    table of 2^clamp(hashLog, 8, 12) positions             minMatch   4..7 (3 is refused by zg_cctx_set_parameter)
//   windowLog  matches no further back than min(2^windowLog, 65535)
// chainLog and targetLength have no counterpart here and are refused when set (zg_cctx_set_parameter).
// A negative level is libzstd's fast strategy with targetLength = -level, which also turns literal compression off:
// Raw literals, and from -2 down the strided parse of ze_fast_block (level -1 keeps level 1's greedy parse: libzstd
// steps only from targetLength 2).  An explicit strategy >= 2 or searchLog asks for another strategy than fast, and
// then a negative level resolves as level 1 does.
static ZeParams ze_resolve_params(const ZgCParams& cp) {
	ZeParams p;
	int level = cp.level;
	const bool fast = level < 0 && cp.strategy < 2 && cp.search_log == 0;
	p.accel = fast ? (u32)zg_min<int>(-level, (int)ZE_ACCEL_MAX) : 0u;
	p.raw_lit = fast ? 1u : 0u;
	if (level < 0) level = 1;
	p.lazy = level >= 3 ? 1 : 0;
	p.ways = level >= 9 ? 4 : level >= 6 ? 2 : 1;
	if (cp.strategy > 0) {
		p.lazy = cp.strategy >= 3 ? 1 : 0;
		p.ways = cp.strategy >= 6 ? 4 : 1;
	}
	if (cp.search_log > 0) p.ways = cp.search_log >= 2 ? 4 : 2;
	p.min_match = cp.min_match >= 4 ? (u32)zg_min<int>(cp.min_match, 7) : ZE_MINMATCH;
	p.max_dist = cp.window_log > 0 && cp.window_log < 16 ? (1u << cp.window_log) : 65535u;
	p.hlog_cap = cp.hash_log > 0 ? (u32)zg_max<int>(8, zg_min<int>(cp.hash_log, ZE_HLOG_MAX)) : (u32)ZE_HLOG_MAX;
	return p;
}

size_t zg_zstd_encode_run(cudaStream_t s, ZgZeWork& w, const u8* blob, const u64* file_off, const u64* comp_off, const u64* file_len,
                          const u32* ulist, const u64* blk_base, u32 nuniq, u64 nblocks, u64 comp_bytes, u8* comp, u32* blk_csize,
                          const ZgCParams& cparams) {
	if (nblocks == 0) return 0;
	const u64 chunk_bytes = g_ze_chunk_bytes;
	u32 nchunks = (u32)((comp_bytes + chunk_bytes - 1) / chunk_bytes);
	if (nchunks == 0) nchunks = 1;
	u64 span = zg_min<u64>(comp_bytes, chunk_bytes) + ZS_BLOCK_MAX + 64;  // a chunk's last block may stick out
	u32 sms = (u32)zg_sm_count();
	u32 grid_m = (u32)zg_min<u64>((nblocks + ZE_WARPS - 1) / ZE_WARPS, (u64)sms * ZE_MIN_CTAS);
	u32 grid_e = (u32)zg_min<u64>((nblocks + ZE_WARPS - 1) / ZE_WARPS, (u64)sms * ZE_ENT_CTAS);
	size_t qbytes = (size_t)nchunks * ZE_NQ * 4 + 16;
	if (w.queue.reserve(qbytes) || w.meta.reserve(nblocks * sizeof(ZeBlkMeta)) || w.seqbuf.reserve(span * 2) || w.litbuf.reserve(span) ||
	    w.codebuf.reserve(span) || w.stbbuf.reserve(span * 2) || w.bounds.reserve(((size_t)nchunks + 1) * 8))
		return ZG_ERR(ZG_error_memory_allocation);
	const bool sorted = nblocks > 8 && nblocks < 0xffffffffull;
	if (sorted && (w.bins.reserve((size_t)nchunks * ZE_OBINS * 4) || w.order.reserve(nblocks * 4) || w.info.reserve(nblocks * sizeof(ZeBlk))))
		return ZG_ERR(ZG_error_memory_allocation);
	cudaMemsetAsync(w.queue.p, 0, qbytes, s);
	const ZeParams prm = ze_resolve_params(cparams);
	ZeJob J;
	J.blob = blob;
	J.file_off = file_off;
	J.comp_off = comp_off;
	J.file_len = file_len;
	J.ulist = ulist;
	J.blk_base = blk_base;
	J.nuniq = nuniq;
	J.nblocks = nblocks;
	J.comp = comp;
	J.blk_csize = blk_csize;
	J.meta = w.meta.as<ZeBlkMeta>();
	J.seqbuf = w.seqbuf.as<u64>();
	J.litbuf = w.litbuf.as<u8>();
	J.codebuf = w.codebuf.as<u32>();
	J.stbbuf = w.stbbuf.as<u64>();
	J.bounds = w.bounds.as<u64>();
	J.order = nullptr;
	J.info = nullptr;
	J.chunk_bytes = chunk_bytes;
	size_t smem_m = sizeof(ZeMatchWarp) * ZE_WARPS;
	size_t smem_l = sizeof(ZeWarp) * ZE_WARPS;
	size_t smem_q = sizeof(ZeWarp) * ZE_WARPS + sizeof(ZePredef);
	static ZgPerDevice attr_dev;
	bool& attr_set = *attr_dev.slot();
	if (!attr_set) {
		if (cudaFuncSetAttribute(k_zstd_match_blocks<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m) != cudaSuccess ||
		    cudaFuncSetAttribute(k_zstd_match_blocks<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m) != cudaSuccess ||
		    cudaFuncSetAttribute(k_zstd_match_blocks<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m) != cudaSuccess ||
		    cudaFuncSetAttribute(k_zstd_match_blocks<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m) != cudaSuccess ||
		    cudaFuncSetAttribute(k_zstd_literals, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_l) != cudaSuccess ||
		    cudaFuncSetAttribute(k_zstd_sequences, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_q) != cudaSuccess)
			return ZG_ERR(ZG_error_device);
		attr_set = true;
	}
	zg_prof_begin(ZG_K_ENCODE, s);
	ZG_LAUNCH(k_ze_chunk_bounds, (nchunks + 128) / 128, 128, 0, s, J, nchunks, w.bounds.as<u64>());
	ZG_COUNT_LAUNCH();
	if (sorted) {
		cudaMemsetAsync(w.bins.p, 0, (size_t)nchunks * ZE_OBINS * 4, s);
		u32 g = (u32)((nblocks + 255) / 256);
		ZG_LAUNCH(k_ze_order_count, g, 256, 0, s, J, nchunks, w.bins.as<u32>());
		ZG_LAUNCH(k_ze_order_scan, nchunks, 32, 0, s, J, w.bins.as<u32>());
		ZG_LAUNCH(k_ze_order_scatter, g, 256, 0, s, J, nchunks, w.bins.as<u32>(), w.order.as<u32>(), w.info.as<ZeBlk>());
		g_zg_launches += 3;
		J.order = w.order.as<u32>();
		J.info = w.info.as<ZeBlk>();
	}
	u32* q = w.queue.as<u32>();
	for (u32 k = 0; k < nchunks; k++) {
		u32* qk = q + (size_t)k * ZE_NQ;
		zg_prof_begin(ZG_K_MATCH, s);
		if (prm.accel >= 2) ZG_LAUNCH(k_zstd_match_blocks<0>, grid_m, ZE_WARPS * 32, smem_m, s, J, k, qk + 0, prm);
		else if (prm.ways == 4) ZG_LAUNCH(k_zstd_match_blocks<4>, grid_m, ZE_WARPS * 32, smem_m, s, J, k, qk + 0, prm);
		else if (prm.ways == 2) ZG_LAUNCH(k_zstd_match_blocks<2>, grid_m, ZE_WARPS * 32, smem_m, s, J, k, qk + 0, prm);
		else ZG_LAUNCH(k_zstd_match_blocks<1>, grid_m, ZE_WARPS * 32, smem_m, s, J, k, qk + 0, prm);
		zg_prof_end(ZG_K_MATCH, s);
		zg_prof_begin(ZG_K_LITERALS, s);
		ZG_LAUNCH(k_zstd_literals, grid_e, ZE_WARPS * 32, smem_l, s, J, k, qk + 1, prm.raw_lit);
		zg_prof_end(ZG_K_LITERALS, s);
		zg_prof_begin(ZG_K_SEQUENCES, s);
		ZG_LAUNCH(k_zstd_sequences, grid_e, ZE_WARPS * 32, smem_q, s, J, k, qk + 2);
		zg_prof_end(ZG_K_SEQUENCES, s);
		g_zg_launches += 3;
	}
	zg_prof_end(ZG_K_ENCODE, s);
	return cudaGetLastError() == cudaSuccess ? 0 : ZG_ERR(ZG_error_device);
}

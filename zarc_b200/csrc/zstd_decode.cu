// K5 + K6: Zstandard frame decode (RFC 8878).  Replaces DCtx::decompress_stream as driven by
// crates/zarc/src/decode/zstd_iterator.rs:88-153 (one frame per content entry, decode/frame_iterator.rs).
//
// One warp owns a batch of 32 frames, ONE FRAME PER LANE.  Everything that is inherently serial
// inside a frame -- frame/block header parsing, the FSE sequence bitstream with its three states,
// repeat-offset resolution -- runs lane-per-frame, so 32 serial chains advance per warp instruction.
// Everything that is parallel inside a frame is done by the whole warp for one frame at a time:
// Huffman/FSE table construction, the 4 literal streams, and sequence execution (literal and match
// copies straight into the frame's output in HBM).
//
// A batch proceeds in rounds, one block per live frame and round:
//   A. per frame (warp-cooperative): block header (Raw/RLE blocks are copied on the spot), literals
//      and sequences section headers, FSE decode tables into the lane's global slot, bitstream init;
//   B. lock-step (lane-per-frame): every lane decodes ALL sequences of its block, resolves repeat
//      offsets and appends them, packed to 8 bytes (offset:28 | litLength:18 | matchLength:18), to
//      the frame's span of the warp's sequence arena;
//   C. per frame (warp-cooperative): Huffman table + the literal streams into the warp's literal
//      buffer, then the sequences are executed 32 at a time -- so while a frame is being written its
//      literals, its sequences and its recent output (the match sources) are cache-hot.
// Blocks of a frame stay in order, so Treeless literals, Repeat_Mode tables, repeat offsets and
// cross-block matches (all produced by libzstd at levels 1/3/9, SURVEY.md App. E) work.  State that
// must outlive a round lives in global scratch: the FSE tables (fixed slot per lane) and where the
// last Huffman tree description is (Treeless blocks read it again).  A block whose sequences do not fit
// the arena waits for the next round.
// HBM traffic: C read + N written (+ 8 B per sequence and the literals staged through L2).
//
// This kernel takes the single-block frames (every file up to 128 KiB: almost all of a source tree) and whatever the
// staged pipeline's header walk refused (the serial decode names the error).  Frames of two blocks and more go through
// the staged pipeline (zstd_decode_staged.cu): all their blocks entropy-decoded in parallel, then executed in block
// order.  Items are handed out largest first, one atomicAdd per batch.
// The uniform per-block helpers (table builds, literals, warp copies) are kept OUT OF LINE on purpose: inlined,
// the kernel was 207 KB of code with 700 B of spills and 12 % slower.
#include "zstd_decode.cuh"
#ifndef ZD_B_STEPS
#define ZD_B_STEPS 64   // sequences a lane decodes before the warp reconverges (phase B)
#endif

// ---------------------------------------------------------------------------------------------
// Frames are handed to the warps in descending order of compressed size (counting sort), so that the
// 32 frames of a batch carry similar numbers of sequences (phase B runs in lock-step) and the big
// frames start first.
#define ZD_BINS 4096u
ZG_DEV u32 zd_bin(u64 len) { return ZD_BINS - 1u - (u32)zg_min<u64>(len >> 4, ZD_BINS - 1u); }
// (`list`: the frames to decode, or null for all of them; an item t is frame list[t])
__global__ void __launch_bounds__(256) k_zd_bin_count(const u64* __restrict__ len, const u32* __restrict__ list, u64 n, u32* bins) {
	u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (t < n) atomicAdd(&bins[zd_bin(len[list ? list[t] : t])], 1u);
}
__global__ void __launch_bounds__(1024) k_zd_bin_scan(u32* bins) {
	// exclusive scan of ZD_BINS counters by one CTA (4 per thread)
	__shared__ u32 part[32];
	u32 t = threadIdx.x, lane = t & 31, w = t >> 5;
	u32 v[4], sum = 0;
	for (u32 i = 0; i < 4; i++) {
		v[i] = bins[4 * t + i];
		sum += v[i];
	}
	u32 incl = zg_warp_incl_scan(sum);
	if (lane == 31) part[w] = incl;
	__syncthreads();
	if (w == 0) {
		u32 p = part[lane];
		u32 pi = zg_warp_incl_scan(p);
		part[lane] = pi - p;
	}
	__syncthreads();
	u32 run = part[w] + incl - sum;
	for (u32 i = 0; i < 4; i++) {
		bins[4 * t + i] = run;
		run += v[i];
	}
}
__global__ void __launch_bounds__(256) k_zd_bin_scatter(const u64* __restrict__ len, const u32* __restrict__ list, u64 n, u32* bins, u32* perm) {
	u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (t < n) perm[atomicAdd(&bins[zd_bin(len[list ? list[t] : t])], 1u)] = (u32)t;
}

// ---------------------------------------------------------------------------------------------
// Huffman literals of the single-block frames, decoded ahead of the fused kernel (which then only copies them): in the
// fused kernel the tree and the streams of a block ran on 1-4 lanes while the rest of the warp waited, frame after frame.
// Here one warp takes a group of ZD_HL_SECS sections (largest first, so that the streams of a group end together):
//  1. trees, one lane per section: the lane reads its section's tree description into its own row of weights (FSE-coded
//     weights through a lane-private table), checks the tree and the jump table, and finds where each weight's entries
//     start in the table;
//  2. tables, warp-wide, a round at a time: a round is as many of the next sections as have their tables fit in
//     ZD_HL_TAB entries (1 << maxbits each) and their streams in 32 lanes.  Each symbol's start in its table is its
//     weight's start plus the entries of the symbols of that weight before it (match_any over 32 symbols at a time);
//  3. the round's streams, one per lane (numbered by a prefix over the sections' stream counts).
// Bytes go to stage + lit_off[s]; lit_at[frame] = lit_off[s], or ZD_LIT_BAD where the fused kernel would have failed the
// section (bad tree, table, jump table, or a stream that does not end exactly).
// Tables per round against warps per SM (one CTA per SM; NVIDIA B200 at 1000 W, 10.2 GB of C2, `tools/kbench.py --what
// pack`, ms of the pre-pass with its sort and scan, all in one call): 16384 entries x 4 warps 21.5 ms, 16384 x 5 18.0,
// 8192 x 8 12.1 (twice), 6144 x 10 11.5; the warp-wide version before (2 sections x 4 warps, 16 warps per SM) 23.5.
// 6144 x 10 was measured once, so the defaults stay at 8192 x 8.  More warps per SM is what moved it; which phase
// bounds it now is not measured.
#ifndef ZD_HL_SECS
#define ZD_HL_SECS 32   // sections per warp and group (1..32)
#endif
#ifndef ZD_HL_WARPS
#define ZD_HL_WARPS 8   // warps per CTA
#endif
#ifndef ZD_HL_TAB
#define ZD_HL_TAB 8192  // u16 table entries per warp and round: 4 sections at maxbits 11, more at fewer bits
#endif
#define ZD_HL_ROW 284u  // bytes per lane: weights (<= 256 symbols), then u16 start per weight [12]; 71 words, so that
                        // the lanes' rows start in different banks
#define ZD_HL_FSE 65u   // u32 per lane of FSE weight table (64 cells), in the table space before the tables are filled
#define ZD_HL_SMEM (32 * ZD_HL_ROW + 32 + ZD_HL_TAB * 2)  // per warp: rows, stream owners, tables
static_assert(ZD_HL_SECS >= 1 && ZD_HL_SECS <= 32, "one lane per section");
static_assert(ZD_HL_TAB >= 2048 && ZD_HL_TAB * 2 >= 32 * ZD_HL_FSE * 4 && ZD_HL_TAB % 8 == 0, "ZD_HL_TAB");

__global__ void __launch_bounds__(ZD_HL_WARPS * 32)
k_zd_huf_literals(const u8* __restrict__ archive, const u64* __restrict__ sec_at, const u32* __restrict__ sec_frame,
                  const u64* __restrict__ lit_off, u64 nsec, const u32* __restrict__ perm, u32* queue, u8* stage, u64* lit_at) {
	ZG_DYN_SMEM(u8, sm);
	u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	u8* rows = sm + warp * ZD_HL_SMEM;
	u8* owner = rows + 32 * ZD_HL_ROW;        // [32]: the section of each stream lane in the round
	u16* tabs = (u16*)(owner + 32);           // ZD_HL_TAB entries
	u8* row = rows + lane * ZD_HL_ROW;
	for (;;) {
		u32 base = 0;
		if (lane == 0) base = atomicAdd(queue, (u32)ZD_HL_SECS);
		base = __shfl_sync(ZG_FULL, base, 0);
		if (base >= nsec) break;
		u32 ng = (u32)zg_min<u64>(ZD_HL_SECS, nsec - base);
		// 1. my section's tree
		u32 si = 0, regen = 0, streams = 0, nw = 0, bits = 0;
		u64 lo = 0;
		const u8 *lp = archive, *lend = archive;
		if (lane < ng) {
			si = perm ? perm[base + lane] : base + lane;
			lo = lit_off[si];
			const u8* src = archive + sec_at[si];
			ZdLitHdr h;
			zd_lit_header(src, ZS_BLOCK_MAX, h);  // validated by the walk (k_zds_count)
			lp = src + h.hdr;
			lend = lp + h.comp;
			regen = h.regen;
			u32 used = zd_read_huf_weights_lane(lp, h.comp, row, (u32*)tabs + lane * ZD_HL_FSE, (u32*)row, &nw);
			bits = used ? zd_huf_weights_check(row, nw, (u16*)(row + 256)) : 0;
			lp += used;
			const u8* sp;
			u32 sn, first, cnt;
			if (bits && zd_huf_split(lp, lend, regen, h.streams, 0, sp, sn, first, cnt)) streams = h.streams;
			else lit_at[sec_frame[si]] = ZD_LIT_BAD;
		}
		__syncwarp();  // (the FSE tables are in the space of the Huffman tables)
		u32 r0 = 0;
		while (r0 < ng) {
			// the round: sections r0.. while their tables and streams fit (a section with a bad tree takes neither)
			u32 mine = lane >= r0 && streams ? (1u << bits) | streams << 20 : 0;
			u32 incl = zg_warp_incl_scan(mine);
			u32 r1 = r0 + (u32)__popc(__ballot_sync(ZG_FULL, lane >= r0 && lane < ng && (incl & 0xfffffu) <= ZD_HL_TAB && (incl >> 20) <= 32));
			ZD_SCHED_COUNT(1);
			bool in = lane >= r0 && lane < r1 && streams;
			u32 toff = (incl & 0xfffffu) - (mine & 0xfffffu), pre = (incl >> 20) - streams;
			// 2. tables
			for (u32 k = r0; k < r1; k++) {
				u32 kb = __shfl_sync(ZG_FULL, in ? bits : 0, k), knw = __shfl_sync(ZG_FULL, nw, k) + 1, kt = __shfl_sync(ZG_FULL, toff, k);
				if (!kb) continue;
				u8* kw = rows + k * ZD_HL_ROW;
				zd_huf_fill_table(tabs + kt, kw, knw, (u16*)(kw + 256), kb);
			}
			// 3. streams
			if (in)
				for (u32 j = 0; j < streams; j++) owner[pre + j] = (u8)lane;
			__syncwarp();
			u32 nst = __shfl_sync(ZG_FULL, incl >> 20, r1 - 1);
			u32 k = lane < nst ? owner[lane] : 0;
			const u8 *kp = zd_bc(lp, k), *ke = zd_bc(lend, k);
			u32 kreg = __shfl_sync(ZG_FULL, regen, k), kst = __shfl_sync(ZG_FULL, streams, k), kb = __shfl_sync(ZG_FULL, bits, k);
			u32 kt = __shfl_sync(ZG_FULL, toff, k), kpre = __shfl_sync(ZG_FULL, pre, k);
			u64 klo = __shfl_sync(ZG_FULL, lo, k);
			bool ok = true;
			if (lane < nst) {
				const u8* sp;
				u32 sn, first, cnt;
				zd_huf_split(kp, ke, kreg, kst, lane - kpre, sp, sn, first, cnt);  // (checked in 1.)
				ok = zd_huf_stream(tabs + kt, kb, sp, sn, stage + klo + first, cnt);
			}
			u32 bad = __ballot_sync(ZG_FULL, !ok);
			if (in) lit_at[sec_frame[si]] = (bad >> pre) & ((1u << streams) - 1u) ? ZD_LIT_BAD : lo;
			__syncwarp();
			r0 = r1;
		}
	}
}

__global__ void __launch_bounds__(ZD_WARPS * 32, ZD_MIN_CTAS)
k_zstd_decode_frames(const u8* __restrict__ archive, u64 archive_len, const u64* __restrict__ off, const u64* __restrict__ len,
                     const u64* __restrict__ ulen, const u64* __restrict__ out_off, u64 nframes, u8* out, u64 out_cap,
                     const u32* __restrict__ perm, const u32* __restrict__ list, u64* seq_arenas, u8* litbufs, u32* tabs, ZdHufSave* hufsaves, u32* queue,
                     u32* status, u64* produced, u32* cksums, u32 cap_div, u32 min_batch, u32 floor_bytes, u32 share_q,
                     const u8* __restrict__ lit_stage, const u64* __restrict__ lit_at) {
	ZG_DYN_SMEM(ZdWarp, sm);
	u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	ZdWarp* W = &sm[warp];
	size_t gw = (size_t)blockIdx.x * ZD_WARPS + warp;
	u64* arena = seq_arenas + gw * ZD_SEQ_ARENA;
	u8* litbuf = litbufs + gw * ZD_LITBUF;
	u32* my_slot = tabs + (gw * 32 + lane) * ZD_TAB_SLOT;
	ZdHufSave* hufsave = hufsaves + gw * 32;
	u64 hint_len = ~0ull;  // compressed size of the last item of this warp's previous batch
	u64 prev_base = 0;
	for (;;) {
		// Hand-out: frames come largest first.  A batch is up to 32 frames, but (a) no more than about
		// ZD_BATCH_BYTES of compressed input -- the phases around the lane-parallel sequence decode run
		// frame after frame, so 32 of the largest frames in one warp would be the kernel's tail --
		// and (b) smaller towards the end, so that the last round is spread over all warps.
		u32 base = 0, want = 32;
		if (lane == 0) {
			// The batch size comes from the size of the last item this warp saw (items come largest first, so it
			// bounds every later one) and from this warp's previous position in the queue: nothing has to be read
			// before the claim, and the claim is one atomicAdd -- no compare-and-swap loop for ~3000 warps to fight over.
			u64 flen = hint_len;
			if (flen == ~0ull) {
				u32 t0 = perm ? perm[0] : 0u;
				flen = len[list ? list[t0] : t0];
			}
			u64 left = nframes > prev_base ? nframes - prev_base : 1;
			u64 share = 4 * left / ((u64)share_q * gridDim.x * ZD_WARPS);  // share_q quarters of ... (8: half a fair share)
			// a quarter of a warp's fair share of the input, but at least min_batch bytes
			u64 cap = zg_max<u64>(min_batch, archive_len / ((u64)cap_div * gridDim.x * ZD_WARPS));
			u64 fit = cap / (flen ? flen : 1);
			// ... and never so small that claiming a batch costs as much as decoding it (the smallest
			// frames come last: they always go out as full rows)
			u64 floor_b = floor_bytes / (flen ? flen : 1);
			want = (u32)zg_min<u64>(zg_min<u64>(32, zg_max<u64>(zg_max<u64>(4, share), floor_b)), zg_max<u64>(2, fit));
			base = atomicAdd(queue, want);
		}
		base = __shfl_sync(ZG_FULL, base, 0);
		want = __shfl_sync(ZG_FULL, want, 0);
		if (base >= nframes) break;
		prev_base = base;
		bool mine = lane < want && (u64)base + lane < nframes;
		u64 t = mine ? (perm ? (u64)perm[base + lane] : (u64)base + lane) : 0;  // work item
		u64 k = (mine && list) ? (u64)list[t] : t;                              // its frame
		// ---- lane-private frame header ----
		ZdLane L;
		L.src = archive;
		L.out = out;
		L.n = L.ip = L.cap = L.opos = L.fcs = L.base = 0;
		L.status = ZS_OK;
		L.flags = 0;
		L.fcs_len = L.cksum = 0;
		L.seq.rep0 = 1;
		L.seq.rep1 = 4;
		L.seq.rep2 = 8;
		L.ll_log = L.ml_log = L.of_log = 0;
		L.blk = archive;
		L.blk_n = L.nseq = L.seq.left = L.seq_base = 0;
		L.seq.b.start = L.seq.b.ptr = archive;
		L.seq.b.lo = L.seq.b.hi = L.seq.b.consumed = 0;
		L.seq.sl = L.seq.so = L.seq.sm = 0;
		u64 mylen = 0;
		if (mine) {
			u64 fo = off[k], fl = len[k], ul = ulen[k], oo = out_off[k];
			mylen = fl;
			if (fo > archive_len || fl > archive_len - fo) L.status = ZS_E_SRC_SIZE;
			else if (oo > out_cap || ul > out_cap - oo) L.status = ZS_E_DST_SMALL;
			else {
				L.src = archive + fo;
				L.n = fl;
				L.out = out + oo;
				L.cap = ul;
				L.flags = ZD_F_ACTIVE;
				ZdFrameHdr F;
				u32 st = zd_frame_header(L.src, L.n, F);
				if (st != ZS_OK) zd_fail(L, st);
				else {
					L.ip = F.ip;
					L.fcs = F.fcs;
					L.fcs_len = F.fcs_len;
					if (F.cksum) L.flags |= ZD_F_CKSUM;
				}
				u64 a = lit_at[k];
				if (a == ZD_LIT_BAD) L.flags |= ZD_F_LIT_BAD;
				else if (a != ZD_LIT_NONE) {
					L.flags |= ZD_F_LIT_STAGED;
					hufsave[lane].staged = lit_stage + a;
				}
			}
		}
		{
			u32 have = __ballot_sync(ZG_FULL, mine);
			hint_len = __shfl_sync(ZG_FULL, mylen, have ? 31 - __clz((int)have) : 0);
		}
		__syncwarp();
		// ---- rounds: one block per live frame ----
		for (;;) {
			u32 live = __ballot_sync(ZG_FULL, (L.flags & ZD_F_ACTIVE) != 0);
			if (!live) break;
			// A: set up the next block of every live frame
			u32 arena_used = 0;
			u32 todo = live;
			while (todo) {
				int f = __ffs((int)todo) - 1;
				todo &= todo - 1;
				ZdLane U = zd_bcast(L, f);
				zd_setup_frame(W, U, tabs + (gw * 32 + (u32)f) * ZD_TAB_SLOT, arena_used, litbuf, hufsave + f);
				if (lane == (u32)f) L = U;
				__syncwarp();
			}
			// B: every lane decodes its block's sequences (in bounded steps, so the warp reconverges)
			{
				const u32* llt = (L.flags & ZD_F_LL_DEF) ? ZS_LL_DEFAULT_DTABLE : my_slot;
				const u32* mlt = (L.flags & ZD_F_ML_DEF) ? ZS_ML_DEFAULT_DTABLE : my_slot + 512;
				const u32* oft = (L.flags & ZD_F_OF_DEF) ? ZS_OF_DEFAULT_DTABLE : my_slot + 1024;
				ZdSeqPlain plain;
				for (;;) {
					u32 cnt = zg_min<u32>((u32)ZD_B_STEPS, L.seq.left);
					if (!__any_sync(ZG_FULL, cnt > 0)) break;
					if (cnt && !zd_lane_decode(L.seq, plain, cnt, llt, mlt, oft, arena + L.seq_base + (L.nseq - L.seq.left))) zd_fail(L, ZS_E_CORRUPT);
				}
			}
			__syncwarp();
			// C: execute frame after frame
			todo = __ballot_sync(ZG_FULL, (L.flags & ZD_F_ACTIVE) && L.nseq > 0);
			while (todo) {
				int f = __ffs((int)todo) - 1;
				todo &= todo - 1;
				ZdLane U = zd_bcast(L, f);
				zd_exec_block(W, U, arena + U.seq_base, litbuf, hufsave + f);
				if (lane == (u32)f) L = U;
				__syncwarp();
			}
		}
		if (mine) {
			bool ok = L.status == ZS_OK;
			status[k] = L.status;
			produced[k] = ok ? L.opos : 0;
			cksums[2 * k] = ok ? L.cksum : 0;
			cksums[2 * k + 1] = (ok && (L.flags & ZD_F_HAS_CK)) ? 1u : 0u;
		}
		__syncwarp();
	}
}

#ifdef ZG_EMU
u64 g_zd_sched[2];
// the scheduling counters (ZD_SCHED_COUNT) since the last call, then zero
extern "C" void zg_internal_sched_stats(u64 out[2]) {
	for (int i = 0; i < 2; i++) {
		out[i] = g_zd_sched[i];
		g_zd_sched[i] = 0;
	}
}
#endif

// hand-out tuning (see the kernel): a batch holds at most 1/cap_div of a warp's fair share of the input but at least
// min_batch bytes; frames so small that 32 of them stay below floor_bytes always go out as full rows
static u32 g_zd_tune[4] = {4, ZD_BATCH_BYTES, 32u << 10, 8};
extern "C" void zg_internal_set_decode_share(u32 q) { g_zd_tune[3] = q ? q : 8; }
extern "C" void zg_internal_set_decode_batching(u32 cap_div, u32 min_batch, u32 floor_bytes) {
	g_zd_tune[0] = cap_div ? cap_div : 4;
	g_zd_tune[1] = min_batch ? min_batch : ZD_BATCH_BYTES;
	g_zd_tune[2] = floor_bytes ? floor_bytes : (32u << 10);
}

// the nsec sections k_zds_count listed (w.hl_*: nlit bytes in all) -> w.hl_stage, w.lit_at
static size_t zd_huf_literals_launch(cudaStream_t s, ZgZdWork& w, const u8* archive, u64 nsec, u64 nlit) {
	if (nsec >= 0xff000000ull) return ZG_ERR(ZG_error_GENERIC);  // (the queue counter runs past nsec by up to one group per warp)
	if (w.hl_stage.reserve(nlit + 64) || w.hl_perm.reserve(nsec * 4)) return ZG_ERR(ZG_error_memory_allocation);
	zg_prof_begin(ZG_K_HUF_LITERALS, s);
	// largest first (the frames' counting sort, over the sizes), then the sizes -> staging offsets
	u64* sizes = w.hl_off.as<u64>();
	cudaMemsetAsync(w.bins.p, 0, ZD_BINS * 4, s);
	u32 g = (u32)((nsec + 255) / 256);
	ZG_LAUNCH(k_zd_bin_count, g, 256, 0, s, sizes, nullptr, nsec, w.bins.as<u32>());
	ZG_LAUNCH(k_zd_bin_scan, 1, 1024, 0, s, w.bins.as<u32>());
	ZG_LAUNCH(k_zd_bin_scatter, g, 256, 0, s, sizes, nullptr, nsec, w.bins.as<u32>(), w.hl_perm.as<u32>());
	g_zg_launches += 3;
	size_t r = zg_scan_run(s, w.tiles, sizes, nsec, 0, sizes, nullptr);
	if (zg_is_error(r)) return r;
	size_t smem = ZD_HL_SMEM * ZD_HL_WARPS;
	static ZgPerDevice attr_dev;
	bool& attr_set = *attr_dev.slot();
	if (!attr_set) {
		if (cudaFuncSetAttribute(k_zd_huf_literals, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
			return ZG_ERR(ZG_error_device);
		attr_set = true;
	}
	u64 groups = (nsec + ZD_HL_SECS - 1) / ZD_HL_SECS;
	u32 per_sm = (u32)zg_max<size_t>(1, (227u << 10) / smem);
	u32 grid = (u32)zg_min<u64>((groups + ZD_HL_WARPS - 1) / ZD_HL_WARPS, (u64)zg_sm_count() * per_sm);
	ZG_LAUNCH(k_zd_huf_literals, grid, ZD_HL_WARPS * 32, smem, s, archive, w.hl_at.as<u64>(), w.hl_frame.as<u32>(), sizes, nsec,
	          w.hl_perm.as<u32>(), w.queue.as<u32>() + 1, w.hl_stage.as<u8>(), w.lit_at.as<u64>());
	ZG_COUNT_LAUNCH();
	zg_prof_end(ZG_K_HUF_LITERALS, s);
	return cudaGetLastError() == cudaSuccess ? 0 : ZG_ERR(ZG_error_device);
}

// one launch of the fused kernel over `count` frames (those in `list`, or all when it is null), handed out largest first,
// after the pre-pass over the Huffman literals of the nsec sections k_zds_count listed (nlit bytes).
// Multi-block frames go through the staged pipeline instead (zstd_decode_staged.cu, which also holds zg_zstd_decode_run).
size_t zd_fused_launch(cudaStream_t s, ZgZdWork& w, const u8* archive, u64 archive_len, const u64* off, const u64* len, const u64* ulen,
                       const u64* out_off, const u32* list, u64 count, u8* out, u64 out_cap, u32* status, u64* produced, u32* cksums,
                       u64 nsec, u64 nlit) {
	if (count == 0) return 0;
	if (count >= 0xff000000ull) return ZG_ERR(ZG_error_GENERIC);  // (the queue counter runs past count by up to one batch per warp)
	u64 batches = (count + 31) / 32;
	u32 grid = (u32)zg_min<u64>((batches + ZD_WARPS - 1) / ZD_WARPS, (u64)zg_sm_count() * ZD_MIN_CTAS);
	size_t warps = (size_t)grid * ZD_WARPS;
	if (w.seqs.reserve(warps * ZD_SEQ_ARENA * 8) || w.lit.reserve(warps * ZD_LITBUF) || w.tabs.reserve(warps * 32 * ZD_TAB_SLOT * 4) ||
	    w.hufsave.reserve(warps * 32 * sizeof(ZdHufSave)) || w.queue.reserve(16) || w.bins.reserve(ZD_BINS * 4) || w.perm.reserve(count * 4))
		return ZG_ERR(ZG_error_memory_allocation);
	cudaMemsetAsync(w.queue.p, 0, 16, s);
	const u32* perm = nullptr;
	if (count > 64) {
		cudaMemsetAsync(w.bins.p, 0, ZD_BINS * 4, s);
		u32 g = (u32)((count + 255) / 256);
		ZG_LAUNCH(k_zd_bin_count, g, 256, 0, s, len, list, count, w.bins.as<u32>());
		ZG_LAUNCH(k_zd_bin_scan, 1, 1024, 0, s, w.bins.as<u32>());
		ZG_LAUNCH(k_zd_bin_scatter, g, 256, 0, s, len, list, count, w.bins.as<u32>(), w.perm.as<u32>());
		g_zg_launches += 3;
		perm = w.perm.as<u32>();
	}
	size_t smem = sizeof(ZdWarp) * ZD_WARPS;
	static ZgPerDevice attr_dev;
	bool& attr_set = *attr_dev.slot();
	if (!attr_set) {
		if (cudaFuncSetAttribute(k_zstd_decode_frames, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
			return ZG_ERR(ZG_error_device);
		attr_set = true;
	}
	zg_prof_begin(ZG_K_DECODE, s);
	if (nsec) {
		size_t r = zd_huf_literals_launch(s, w, archive, nsec, nlit);
		if (zg_is_error(r)) return r;
	}
	ZG_LAUNCH(k_zstd_decode_frames, grid, ZD_WARPS * 32, smem, s, archive, archive_len, off, len, ulen, out_off, count, out, out_cap,
	          perm, list, w.seqs.as<u64>(), w.lit.as<u8>(), w.tabs.as<u32>(), w.hufsave.as<ZdHufSave>(), w.queue.as<u32>(), status, produced, cksums,
	          g_zd_tune[0], g_zd_tune[1], g_zd_tune[2], g_zd_tune[3], w.hl_stage.as<u8>(), w.lit_at.as<u64>());
	zg_prof_end(ZG_K_DECODE, s);
	ZG_COUNT_LAUNCH();
	return cudaGetLastError() == cudaSuccess ? 0 : ZG_ERR(ZG_error_device);
}

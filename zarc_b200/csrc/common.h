// Internal declarations shared by the kernels' launchers and the C ABI.
#pragma once
#include <atomic>
#include "simt.h"
#include "../../include/zarcgpu.h"

#define ZG_ERR(code) ((size_t)0 - (size_t)(code))

extern uint64_t g_zg_slice_bytes, g_zg_pack_slice_bytes;  // host-buffer API: bytes per pipelined slice, unpack / pack (tests shrink them)
extern std::atomic<uint64_t> g_zg_launches;  // kernels launched by this library (bench.py's gpu_launches)
#define ZG_COUNT_LAUNCH() (++g_zg_launches)

// grow-only device buffer
struct ZgBuf {
	void* p = nullptr;
	size_t cap = 0;
	cudaError_t reserve(size_t n) {
		if (n <= cap) return cudaSuccess;
		if (p) cudaFree(p);
		p = nullptr;
		cap = 0;
		size_t want = n + n / 8 + 256;
		cudaError_t e = cudaMalloc(&p, want);
		if (e == cudaSuccess) cap = want;
		return e;
	}
	void release() {
		if (p) cudaFree(p);
		p = nullptr;
		cap = 0;
	}
	template <typename T>
	T* as() const { return (T*)p; }
};
struct ZgHostBuf {  // grow-only pinned host buffer
	void* p = nullptr;
	size_t cap = 0;
	cudaError_t reserve(size_t n) {
		if (n <= cap) return cudaSuccess;
		if (p) cudaFreeHost(p);
		p = nullptr;
		cap = 0;
		size_t want = n + n / 8 + 256;
		cudaError_t e = cudaMallocHost(&p, want);
		if (e == cudaSuccess) cap = want;
		return e;
	}
	void release() {
		if (p) cudaFreeHost(p);
		p = nullptr;
		cap = 0;
	}
	template <typename T>
	T* as() const { return (T*)p; }
};

int zg_sm_count();
// function attributes (opt-in shared memory) are per device: one flag per device, not one per process
struct ZgPerDevice {
	bool done[64] = {};
	bool* slot() {
		static bool never = false;
		int d = 0;
		if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return &(never = false);
		return &done[d];
	}
};

// ---- blake3.cu ----
struct ZgB3Work {
	ZgBuf cnt, cbase, tiles;  // chunks per file, their exclusive prefix (+ the total), scan scratch
	ZgBuf meta;               // u64: chunks in all, end of the data, chunks of the largest file
	ZgBuf taskfile;           // u32 per group of 32 chunks: the file of its first chunk
	ZgBuf cv0, cv1;           // chaining values: chunks / tree levels (ping-pong)
	ZgBuf ltab;               // u32 per block of every tree level: the file of its first slot
	ZgHostBuf h;              // pinned: meta for the host
};
size_t zg_blake3_run(cudaStream_t s, ZgB3Work& w, const u8* blob, const u64* off, const u64* len, u64 n, u8* digests);
void zg_b3work_free(ZgB3Work& w);

// ---- xxh64.cu ----
size_t zg_xxh64_run(cudaStream_t s, const u8* blob, const u64* off, const u64* len, u64 n, u64* hashes);

// ---- corpus.cu ----
size_t zg_corpus_run(cudaStream_t s, u8* out, const u64* seg_off, const u32* seg_len, const u8* seg_kind, const u64* seg_key, u64 nseg);

// ---- scan.cu ----
size_t zg_scan_run(cudaStream_t s, ZgBuf& tiles, const u64* in, u64 n, u64 base, u64* out, u64* total_out);
cudaError_t zg_publish(cudaStream_t s, const void* dev_src, void* pinned_dst, u32 nbytes);  // small results -> pinned host memory, no copy engine

// ---- zstd_decode.cu ----
struct ZgZdStaged {  // the staged pipeline for multi-block frames (zstd_decode_staged.cu)
	ZgBuf nblk, first, multi, single, tot, hist;                 // per frame: block count, first block; frame lists; totals; histogram
	ZgBuf blk, res, out_pos, rep_in, dep, done;                  // per block
	ZgBuf tail, f_out, f_rep, f_status, done_upto, f_chain;      // per frame: running state across chunks
	ZgBuf item_of, chain_list;                                   // per block: its item in the chunk; frames for the chain executor
	ZgBuf jbase, cursor, queue, items, seq_cnt, lit_cnt, seq_off, lit_off, seq_stage, lit_stage, tabs;  // per chunk
	// Content_Checksum of the staged frames, hashed chunk by chunk on a side stream while the next chunk decodes:
	// per frame the KiB chunks hashed so far and the four accumulators; the watermark snapshot of the chunk being hashed
	ZgBuf xx_done, xx_acc, xx_wm;
	u64 xx_n = 0;  // frames the state arrays of the last run cover (0: none)
	cudaStream_t xx_stream = nullptr;
	cudaEvent_t xx_fork = nullptr, xx_join = nullptr;
	bool xx_init = false;
	ZgHostBuf hh;
	void release() {
		for (ZgBuf* b : {&nblk, &first, &multi, &single, &tot, &hist, &blk, &res, &out_pos, &rep_in, &dep, &done, &tail, &f_out, &f_rep, &f_status,
		                 &done_upto, &f_chain, &item_of, &chain_list, &jbase, &cursor, &queue, &items, &seq_cnt, &lit_cnt, &seq_off, &lit_off, &seq_stage, &lit_stage, &tabs, &xx_done, &xx_acc, &xx_wm})
			b->release();
		hh.release();
		if (xx_stream) cudaStreamDestroy(xx_stream);
		if (xx_fork) cudaEventDestroy(xx_fork);
		if (xx_join) cudaEventDestroy(xx_join);
		xx_stream = nullptr;
		xx_fork = xx_join = nullptr;
		xx_init = false;
		xx_n = 0;
	}
};
struct ZgZdWork {
	ZgBuf seqs;     // per-warp sequence arenas
	ZgBuf lit;      // per-warp literal buffers
	ZgBuf tabs;     // per-lane FSE decode-table slots
	ZgBuf hufsave;  // per-lane ZdHufSave: where the last Huffman tree description (Treeless blocks) and staged literals are
	ZgBuf queue;    // frame queue counter
	ZgBuf bins, perm;  // size-sorted hand-out order
	ZgBuf tiles;       // scan scratch
	// Huffman literals of the single-block frames, decoded ahead (k_zd_huf_literals): per section its archive offset,
	// frame, size (then staging offset) and hand-out order; the staged bytes; per frame where its literals are (lit_at)
	ZgBuf hl_at, hl_frame, hl_off, hl_perm, hl_stage, lit_at;
	ZgZdStaged st;
	ZgHostBuf h;
	void release() {
		for (ZgBuf* b : {&seqs, &lit, &tabs, &hufsave, &queue, &bins, &perm, &tiles, &hl_at, &hl_frame, &hl_off, &hl_perm, &hl_stage, &lit_at})
			b->release();
		st.release();
		h.release();
	}
};
size_t zg_zstd_decode_run(cudaStream_t s, ZgZdWork& w, const u8* archive, u64 archive_len, const u64* off, const u64* len,
                          const u64* ulen, const u64* out_off, u64 n, u8* out, u64 out_cap, u32* status, u64* produced,
                          u32* cksums, int verify_checksums = 0);

// ---- glue.cu ----
size_t zg_unpack_finalize_run(cudaStream_t s, const u8* out, const u64* out_off, const u64* ulen, const u64* produced,
                              const u32* cksums, u32* status, u64 n, int verify, const ZgZdWork* zw = nullptr);
size_t zg_verify_spans_run(cudaStream_t s, const u32* status, const u64* out_off, const u64* ulen, u64 out_cap, u64 n, u64* voff, u64* vlen);
size_t zg_digest_compare_run(cudaStream_t s, const u8* got, const u8* want, const u32* status, u8* ok, u64 n);
size_t zg_first_error_run(cudaStream_t s, const u32* status, u64 n, u64* first);

// ---- zstd_encode.cu ----
struct ZgZeWork {
	ZgBuf queue;    // per chunk: per kernel block counters + the table-arena counter
	ZgBuf meta;     // per block: what one kernel hands to the next
	ZgBuf seqbuf, litbuf, codebuf, stbbuf;  // per chunk staging between (and inside) the kernels
	ZgBuf bounds;   // first block of every chunk
	ZgBuf bins, order, info;  // hand-out order of the blocks (per chunk, largest first) and the block -> file table
	void release() {
		for (ZgBuf* b : {&queue, &meta, &seqbuf, &litbuf, &codebuf, &stbbuf, &bounds, &bins, &order, &info}) b->release();
	}
};
struct ZgCParams {  // the cctx's compression parameters (0 = not set), libzstd's names
	int level, window_log, hash_log, search_log, min_match, strategy;
};
size_t zg_zstd_encode_run(cudaStream_t s, ZgZeWork& w, const u8* blob, const u64* file_off, const u64* comp_off, const u64* file_len,
                          const u32* ulist, const u64* blk_base, u32 nuniq, u64 nblocks, u64 comp_bytes, u8* comp, u32* blk_csize,
                          const ZgCParams& cparams);

// ---- per-kernel device timing (abi.cu): CUDA events on the launching stream, off by default ----
enum {
	ZG_K_BLAKE3 = 0, ZG_K_ENCODE = 1 /* the whole encode pass */, ZG_K_DECODE = 2, ZG_K_ASSEMBLE = 3, ZG_K_XXH64 = 4, ZG_K_DEDUP = 5,
	ZG_K_MATCH = 6, ZG_K_LITERALS = 7, ZG_K_SEQUENCES = 8, ZG_K_HUF_LITERALS = 9 /* inside ZG_K_DECODE */, ZG_K_COUNT = 10
};
void zg_prof_begin(int k, cudaStream_t s);
void zg_prof_end(int k, cudaStream_t s);

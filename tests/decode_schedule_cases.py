"""The decoder's scheduling layer: which frames share a warp's batch, a round of its 131 072-entry sequence arena
(ZD_SEQ_ARENA) and a round of the Huffman literals pre-pass's table space (ZD_HL_TAB).  Results must not depend on it, so
every case here is a batch whose bytes, statuses and return code are fixed by the frames alone, run under hand-out
settings that put the frames in different batches and rounds.

Reach is proved by arithmetic, not by the kernel: the sequences of each frame (from its description, equal to what the C
oracle counts) and the hand-out rule give how many block set-ups a batch defers (`arena_defers`); the sections' table
sizes and stream counts give how many rounds the pre-pass takes (`prepass_rounds`).  The emulator build also counts both
events (zg_internal_sched_stats), and its tests check the counts against that arithmetic.

Shared by tests/test_decode_schedule_emu.py and tests/test_decode_schedule_gpu.py."""
import ctypes as C
import functools
import struct

from oracle import ref_path
from tests import handmade_cases as H
from tests import huf_tree_cases as T
from tests import zstd_writer as W
from tests.golden.recipes import text
from tests.helpers import unpack_batch

ARENA = 1 << 17   # ZD_SEQ_ARENA: sequences per warp and round
DENSE = 32_768    # (1, 1, 3) sequences regenerating exactly 128 KiB
MAX_SEQ = 43_690  # the most sequences a 128 KiB block holds (3 bytes each, and one literal)
CORRUPT = 20

# hand-out settings: (name, zg_internal_set_decode_batching arguments or None, zg_internal_set_decode_share argument or
# None, the batch size every warp claims or None when it varies)
SETTINGS = [
    ("want32", (1, 0xFFFFFFFF, 0xFFFFFFFF), None, 32),  # every cap and floor at its largest: 32 frames a batch
    ("want2", (0xFFFFFFFF, 1, 1), None, 2),             # a 1-byte cap: 2 frames a batch
    ("defaults", None, None, None),
    ("share1", None, 1, None),
    ("share_max", None, 0xFFFFFFFF, None),
]


class Item:
    """one frame of a batch: its bytes, what it must restore (None: rejected), its status, and the sequence count of each
    block in order (0 for blocks without sequences; a failing frame lists the blocks up to the one that fails)"""

    def __init__(self, name, frame, want, status=0, nseq=(0,), ulen=None):
        self.name, self.frame, self.want, self.status, self.nseq = name, frame, want, status, list(nseq)
        self.ulen = len(want) if ulen is None else ulen


def _item(name, desc, status=0):
    exp = W.execute(desc) if status == 0 else None
    nseq = [len(b.get("seqs", ())) if b["kind"] == "comp" else 0 for b in desc["blocks"]]
    return Item(name, W.write(desc), exp, status, nseq, W.nominal_size(desc))


def _lit_offset(frame):
    """where the first block's literals section starts (the frame header, then a 3-byte block header)"""
    fhd = frame[4]
    did = {0: 0, 1: 1, 2: 2, 3: 4}[fhd & 3]
    fcs = {0: 1 if fhd & 0x20 else 0, 1: 2, 2: 4, 3: 8}[fhd >> 6]
    return 5 + (0 if fhd & 0x20 else 1) + did + fcs + 3


def _sec_len(sec):
    """bytes of a compressed literals section"""
    sf = (sec[0] >> 2) & 3
    hl, cbits = {0: (3, 10), 1: (3, 10), 2: (4, 14), 3: (5, 18)}[sf]
    return hl + ((int.from_bytes(sec[:hl], "little") >> (4 + cbits)) & ((1 << cbits) - 1))


def huf_section(data, weights=None, streams=4, short=None):
    """a Huffman literals section of data; with `short` = k, stream k codes only the first 8 symbols of its segment, so
    that decoding the segment runs out of bits.  (A stream under 8 bytes also keeps libzstd off its fast 4-stream
    decoder, which does not check where a stream ends: it rejects the section as the RFC asks.)"""
    weights = weights or W.weights_from_data(data)
    code = W.HufCode(weights)
    tree = W.weights_direct(weights) if len(weights) - 1 <= 128 else W.weights_fse(weights)
    if streams == 1:
        body = tree + code.stream(data[:8] if short == 0 else data)
    else:
        seg = (len(data) + 3) // 4
        segs = [data[i * seg : (i + 1) * seg] if i < 3 else data[3 * seg :] for i in range(4)]
        parts = [code.stream(d[:8] if i == short else d) for i, d in enumerate(segs)]
        body = tree + struct.pack("<HHH", *(len(p) for p in parts[:3])) + b"".join(parts)
    return W.lit_header(2, len(data), len(body), streams, 3 if streams == 1 else None) + body


def _swap_literals(frame, sec):
    """the single-block frame with its literals section replaced (and its block size fixed)"""
    at = _lit_offset(frame)
    old = _sec_len(frame[at:])
    bh = int.from_bytes(frame[at - 3 : at], "little")
    bsize = (bh >> 3) - old + len(sec)
    return frame[: at - 3] + struct.pack("<I", (bh & 7) | bsize << 3)[:3] + sec + frame[at + old :]


# ---------------------------------------------------------------------------------------------------------------------
# sequence-dense frames
RLE_TABLES = dict(ll=("rle", 1), of=("rle", 0), ml=("rle", 0))  # (1, 1, 3): literal length 1, rep0 (= 1), match 3


def _dense_desc(lit, n=DENSE):
    return dict(blocks=[H.comp(lit, [(1, 1, 3)] * n, **RLE_TABLES)])


@functools.lru_cache(maxsize=None)
def dense(kind, seed, n=DENSE):
    """n sequences (1, 1, 3) at no bits each: 4 n bytes.  kind "raw": Raw literals; "huf": Huffman literals with a fresh
    tree (decoded ahead by the pre-pass); "huf_bad": the same with a 4th stream that runs out of bits"""
    lits = text(n, seed)
    if kind == "raw":
        return _item(f"dense_raw_{seed}", _dense_desc(H.raw_lit(lits), n))
    it = _item(f"dense_huf_{seed}", _dense_desc(H.huf(lits, streams=4), n))
    if kind == "huf":
        return it
    return Item(f"dense_huf_bad_{seed}", _swap_literals(it.frame, huf_section(lits, short=3)), None, CORRUPT, it.nseq, it.ulen)


def _max_desc(extra_bits=0, first=b"M"):
    # one literal, then 43 690 matches of 3 at distance 1 (an offset of 1 given as a new offset: 2 bits each; the LL table
    # codes 1 once and 0 after it)
    seqs = [W.seq(1, 1, 3)] + [W.seq(0, 1, 3)] * (MAX_SEQ - 1)
    return dict(blocks=[H.comp(H.raw_lit(first), seqs, ll=("fse", 5, [31, -1]), of=("rle", 2), ml=("rle", 0), extra_bits=extra_bits)], fcs=4)


@functools.lru_cache(maxsize=None)
def max_seq(first=b"M"):
    """the most sequences a block can carry: 43 690, regenerating 131 071 bytes"""
    return _item(f"max_seq_{first[0]}", _max_desc(first=first))


@functools.lru_cache(maxsize=None)
def max_seq_bits_left():
    """the same with 3 bits left over after the last sequence: the sequence decode fails, after the set-up has taken its
    arena space.  (2 bits short would not do: the offset bits read past the start are zeros, the values they stand for,
    and libzstd accepts a stream that ends so.)"""
    d = _max_desc(extra_bits=3)
    return Item("max_seq_bits_left", W.write(d), None, CORRUPT, [MAX_SEQ], W.nominal_size(d))


def _small(name, n, seed):
    return _item(name, H.frame(H.comp(H.raw_lit(text(n, seed)))))


EMPTY = lambda: _item("empty", H.frame(dict(kind="raw", data=b"")))  # noqa: E731
BAD_DICT = lambda: Item("dictionary_id", W.write(H.frame(H.comp(H.raw_lit(b"abc")), did=(1, 7))), None, 32, [0], 3)  # noqa: E731


# ---------------------------------------------------------------------------------------------------------------------
# arena cases: (name, items).  Run in this order, so that with 32 frames a batch the frames share one warp lane by lane.
def arena_cases(scale=1):
    """`scale` frames of 43 690 sequences beyond the 8 the cases need at least (the GPU runs more)"""
    fill = [dense("raw", 1), dense("huf", 2), dense("raw", 3), dense("huf", 4)]
    out = [
        ("arena_full", fill),                                   # 4 x 32 768 = 131 072: full, nothing defers
        ("arena_full_plus_one", fill + [dense("huf", 5)]),      # the fifth defers once
        ("arena_bad_literals_deferred", fill + [dense("huf_bad", 6)]),
        ("max_seq_three_a_round", [max_seq(bytes([65 + i])) for i in range(8 * scale)]),
    ]
    mixed = [dense("raw", 7), dense("huf", 8), _small("literals_only", 900, 9), dense("huf_bad", 10), EMPTY(), dense("huf", 11),
             max_seq_bits_left(), dense("raw", 12), BAD_DICT(), _small("literals_only_2", 5000, 13), max_seq(b"Z")]
    out.append(("arena_mixed", mixed))
    out.append(("arena_mixed_reversed", mixed[::-1]))
    return out


def arena_defers(items, want):
    """block set-ups deferred when every warp claims `want` frames in batch order (fewer than 65 frames: no sort).  A
    round sets up the next block with sequences of every live frame, lane by lane, while the arena has room; blocks
    without sequences are finished in the set-up; a failing frame ends after its listed blocks."""
    n = 0
    for b in range(0, len(items), want):
        left = [[k for k in it.nseq] for it in items[b : b + want]]
        while any(left):
            used = 0
            for blocks in left:
                while blocks and blocks[0] == 0:
                    blocks.pop(0)
                if not blocks:
                    continue
                if used + blocks[0] > ARENA:
                    n += 1
                    continue
                used += blocks.pop(0)
    return n


# ---------------------------------------------------------------------------------------------------------------------
# multi-block frames on the lane path: the block with 32 768 sequences of the last four frames waits a round, behind
# the second blocks of the first four (4 x 32 768), and what it needs from the frame's earlier blocks must survive the wait
def lane_path_cases():
    lits = [text(DENSE + 1200, 20 + i) for i in range(9)]
    few = [(1, 1, 3)] * 5
    fill = [H.frame(H.comp(H.raw_lit(lits[i][:5]), few, **RLE_TABLES), H.comp(H.raw_lit(lits[i][:DENSE]), [(1, 1, 3)] * DENSE, **RLE_TABLES))
            for i in range(4)]
    L = lits[4]
    treeless = H.frame(H.comp(H.huf(L[:150], weights=W.weights_from_data(L)), few, **RLE_TABLES),
                       H.comp(H.treeless(L[150 : 150 + DENSE], streams=4), [(1, 1, 3)] * DENSE, **RLE_TABLES))
    s1 = [W.seq(4, 2, 5), (1, 1, 3), W.seq(2, 3, 4), (1, 1, 3), (1, 2, 3)] * 4
    t = H._tables_for(s1 + [(1, 1, 3)])
    L = lits[5]
    repeat_mode = H.frame(H.comp(H.raw_lit(L[:100]), s1, **t), H.comp(H.raw_lit(L[100 : 100 + DENSE]), [(1, 1, 3)] * DENSE, ll="rep", of="rep", ml="rep"))
    L = lits[6]
    # the first block leaves rep0 = 2, rep1 = 1: the second block's matches are at distance 2
    rep_codes = H.frame(H.comp(H.raw_lit(L[:30]), [W.seq(9, 1, 4), W.seq(6, 2, 4)], **dict(ll="pre", of="pre", ml="pre")),
                        H.comp(H.raw_lit(L[30 : 30 + DENSE]), [(1, 1, 3)] * DENSE, **RLE_TABLES))
    L = lits[7]
    raw_rle_before = H.frame(H.comp(H.huf(L[:150], weights=W.weights_from_data(L)), few, **RLE_TABLES), dict(kind="raw", data=L[150:1150]),
                             dict(kind="rle", byte=0x2D, size=700), H.comp(H.treeless(L[1150 : 1150 + DENSE], streams=4), [(1, 1, 3)] * DENSE, **RLE_TABLES))
    descs = [(f"fill_{i}", d) for i, d in enumerate(fill)] + [("deferred_treeless", treeless), ("deferred_repeat_mode", repeat_mode),
                                                              ("deferred_rep_codes", rep_codes), ("deferred_after_raw_rle", raw_rle_before)]
    return descs


@functools.lru_cache(maxsize=None)
def lane_path_items():
    return [_item(n, d) for n, d in lane_path_cases()]


# ---------------------------------------------------------------------------------------------------------------------
# the mixed batch: libzstd frames at levels 1 / 3 / 9 / 19 and this library's frames of the encoder-edge inputs
MIXED_INPUTS = ("raw_headers", "huf_headers", "table_modes", "weights")
MIXED_COUNTS = (1, 31, 33, 64, 65, 97)  # around one warp's batch and the first count the fused launch sorts (> 64)


def mixed_pool(lib):
    from tests import encoder_edge_cases as E

    pool = []
    for name in MIXED_INPUTS:
        datas, _ = E.case_inputs(name)
        for lv in (1, 3, 9, 19):
            pool += [Item(f"{name}.zstd{lv}.{i}", ref_path.ref_compress(d, level=lv), d) for i, d in enumerate(datas)]
        pool += [Item(f"{name}.ours.{i}", f, d) for i, (d, f) in enumerate(zip(datas, E.pack_frames(lib, datas, 3)))]
    return pool


def mixed_batch(pool, count):
    """`count` frames of the pool, taken in a stride that interleaves the inputs and levels"""
    return [pool[(i * 7) % len(pool)] for i in range(count)]


# ---------------------------------------------------------------------------------------------------------------------
# pre-pass rounds.  Each case is at most 32 sections: one group of the default build.  Sections of one shape share a
# Regenerated_Size; different shapes are at least 16 bytes apart (their own bin of the largest-first sort), so that
# the rounds do not depend on the order within a bin.
class Sec:
    def __init__(self, name, section, regen, data, bits, streams):
        self.name, self.section, self.regen, self.data, self.bits, self.streams = name, section, regen, data, bits, streams

    def item(self):
        return Item(self.name, T.frame(self.section, self.regen), self.data, 0 if self.data is not None else CORRUPT, [0], self.regen)


def prepass_items(secs):
    return [s.item() for s in secs]


def _sec(name, data, weights=None, streams=4, short=None):
    weights = weights or W.weights_from_data(data)
    good = short is None
    return Sec(name, huf_section(data, weights, streams, short), len(data), data if good else None, W.HufCode(weights).max_bits, streams)


def _perm(data, seed):
    """the bytes of data in another order (same counts, same tree)"""
    import numpy as np

    a = np.frombuffer(data, dtype=np.uint8).copy()
    np.random.default_rng(seed).shuffle(a)
    return a.tobytes()


W11 = [0] * 97 + [1, 1] + list(range(2, 11)) + [11]  # code lengths 11, 11, 10, ..., 2, 1
D11 = bytes(range(97, 109)) * 3 + b"l" * 900


def bits11(i):
    """a 1-stream section with 11-bit codes (a 2048-entry table), 936 bytes"""
    return _sec(f"bits11_{i}", _perm(D11, i), W11, streams=1)


def small4(i, regen=2000, short=None):
    d = text(regen, 100 + i)
    return _sec(f"s4_{regen}_{i}" + ("" if short is None else f"_short{short}"), d, W.weights_from_data(d, 8), streams=4, short=short)


def small1(i, regen=600, short=None):
    d = text(regen, 300 + i)
    return _sec(f"s1_{regen}_{i}" + ("" if short is None else "_short"), d, W.weights_from_data(d, 8), streams=1, short=short)


def nbits(bits, regen, seed):
    """a 4-stream section whose longest code is exactly `bits` (a uniform spread over 2^(bits-1) + 1 symbols)"""
    k = (1 << (bits - 1)) + 1
    d = _perm(bytes(i % k + 1 for i in range(regen)), seed)
    s = _sec(f"bits{bits}_{regen}", d, W.weights_from_data(d, bits), streams=4)
    assert s.bits == bits, (bits, s.bits)
    return s


def bad_tree(regen, name):
    """a 4-stream section whose tree has a weight of 12"""
    tree = T.direct_tree([12, 1, 1])
    body = tree + b"\x5a" * 60 + b"\x81"
    return Sec(name, W.lit_header(2, regen, len(body), 4, None) + body, regen, None, 0, 0)


def prepass_cases():
    """(name, sections in hand-out order)"""
    out = [
        ("bits11_x4_fills_the_table_space", [bits11(i) for i in range(4)]),
        ("bits11_x5", [bits11(i) for i in range(5)]),
        ("streams4_x8_fill_32_lanes", [small4(i) for i in range(8)]),
        ("streams4_x9", [small4(i) for i in range(9)]),
        ("streams4_x7_and_1_stream_x4", [small4(i) for i in range(7)] + [small1(i) for i in range(4)]),
        ("bits11_x2_and_6", [bits11(0), bits11(1), nbits(6, 800, 1)]),  # 2 x 2048 + 64 = 4160
        ("bits11_x2_and_7", [bits11(0), bits11(1), nbits(7, 800, 1)]),  # 2 x 2048 + 128 = 4224
    ]
    # a bad section first, in the middle and last of a full round (32 streams): a bad tree takes no lanes, a bad stream
    # takes its four
    for what in ("tree", "stream4", "stream1"):
        for where, regen in (("first", 2400), ("middle", 2000), ("last", 1600)):
            n = 8 if what == "tree" else 7
            good = [small4(i, 2200) for i in range(4)] + [small4(i, 1800) for i in range(4, n)]
            bad = bad_tree(regen, f"bad_tree_{where}") if what == "tree" else small4(9, regen, short=3 if what == "stream4" else 0)
            secs = [bad] + good if where == "first" else good[:4] + [bad] + good[4:] if where == "middle" else good + [bad]
            out.append((f"bad_{what}_{where}", secs))
    # a bad 1-stream section among 1-stream ones after seven 4-stream sections (32 streams)
    ones = [small1(i) for i in range(4)]
    out.append(("bad_1_stream_section_in_full_round", [small4(i) for i in range(7)] + ones[:2] + [small1(7, 580, short=0)] + ones[3:4]))
    return out


def prepass_rounds(secs, tab, per_group):
    """rounds of k_zd_huf_literals: groups of `per_group` sections in hand-out order; a round takes the group's next
    sections while their tables (2^bits entries) fit in `tab` and their streams in 32 lanes (a section with a bad tree
    takes neither)"""
    n = 0
    for g in range(0, len(secs), per_group):
        grp = secs[g : g + per_group]
        r0 = 0
        while r0 < len(grp):
            t = s = 0
            r1 = r0
            for x in grp[r0:]:
                t += (1 << x.bits) if x.streams else 0
                s += x.streams
                if t > tab or s > 32:
                    break
                r1 += 1
            n += 1
            r0 = r1
    return n


# ---------------------------------------------------------------------------------------------------------------------
def check_reference(items):
    """libzstd one-shot and streaming and the C oracle restore each valid frame exactly, with the sequence count its
    item lists; each invalid frame is rejected by libzstd's streaming decoder and by the C oracle"""
    for it in items:
        got, err, used, st = ref_path.c_zstd_decompress_frame(it.frame, it.ulen + 64)
        if it.want is None:
            assert H._ref_rejects(it.frame) and err != 0, (it.name, "the reference accepts this frame")
            continue
        assert ref_path.ref_decompress(it.frame, it.ulen + 64) == it.want, (it.name, "libzstd one-shot")
        assert ref_path.ref_decompress_stream(it.frame + b"\x28\xb5\x2f\xfdnext", 0) == it.want, (it.name, "libzstd streaming")
        assert err == 0 and got == it.want and used == len(it.frame), (it.name, "C oracle", err)
        assert st["sequences"] == sum(it.nseq), (it.name, "sequences", st["sequences"], it.nseq)


def _set(lib, batching, share):
    lib.dll.zg_internal_set_decode_batching(*(C.c_uint32(v) for v in (batching or (0, 0, 0))))
    lib.dll.zg_internal_set_decode_share(C.c_uint32(share or 0))


def sched_stats(lib):
    """the emulator build's counters since the last call: (deferred set-ups, pre-pass rounds); None on the product"""
    f = getattr(lib.dll, "zg_internal_sched_stats", None)
    if f is None:
        return None
    out = (C.c_uint64 * 2)()
    f(out)
    return tuple(out)


def run_batch(lib, items, what=""):
    """one zg_unpack_batch of the items: every frame's bytes and status, and the return code naming the first failure
    in batch order"""
    outs, ok, status, rc = unpack_batch(lib, [it.frame for it in items], [it.ulen for it in items],
                                        [ref_path.c_blake3(it.want if it.want is not None else b"") for it in items])
    for j, it in enumerate(items):
        assert status[j] == it.status, (what, it.name, "status", status[j], it.status)
        if it.want is not None:
            assert ok[j] == 1 and outs[j] == it.want, (what, it.name, "bytes differ")
        else:
            assert ok[j] == 0, (what, it.name)
    bad = [it.status for it in items if it.status]
    if bad:
        assert lib.zg_is_error(rc) and lib.zg_get_error_code(rc) == bad[0], (what, "return code", rc)
    else:
        assert rc == 0, (what, rc)


def run_settings(lib, items, what, lane_path=False, settings=SETTINGS):
    """the batch under every hand-out setting (knobs restored afterwards).  Returns {setting: deferred set-ups counted by
    the emulator build} for the settings with a fixed batch size (None on the product)."""
    counted = {}
    try:
        if lane_path:
            lib.dll.zg_internal_set_decode_split_min(C.c_uint64(1 << 40))
        for name, batching, share, want in settings:
            _set(lib, batching, share)
            sched_stats(lib)
            run_batch(lib, items, (what, name))
            st = sched_stats(lib)
            if want is not None:
                counted[name] = None if st is None else st[0]
    finally:
        _set(lib, None, None)
        lib.dll.zg_internal_set_decode_split_min(C.c_uint64(0))
    return counted


def check_arena_case(lib, name, items, lane_path=False):
    """bytes under every setting; the deferrals the arithmetic predicts, and on the emulator build the ones counted"""
    counted = run_settings(lib, items, name, lane_path)
    want = {s: arena_defers(items, w) for s, _, _, w in SETTINGS if w is not None}
    assert want["want2"] == 0, (name, "two frames always fit the arena")
    for s, n in counted.items():
        assert n is None or n == want[s], (name, s, "deferred set-ups", n, want[s])
    return want["want32"]

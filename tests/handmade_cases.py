"""Hand-built Zstandard frames (tests/zstd_writer.py) through every decode path: the shapes libzstd and this library's
encoder rarely or never write -- Repeat_Mode of Predefined / RLE tables, tables and Huffman trees inherited across
blocks without sequences or with Raw / RLE literals, "rep0 - 1" out of an earlier block's history, FSE table descriptions
and Huffman weights at their edges, every header size form -- with the expected bytes computed from the description,
not by a decoder.  Shared by the CPU test-suite (tests/test_handmade_frames_emu.py), the GPU suite and
tools/fuzz_handmade.py.  `handmade_frames` raises AssertionError on the first disagreement and returns counters."""
import ctypes as C

import numpy as np

from oracle import ref_path
from tests import zstd_writer as W
from tests.golden.recipes import rand, text
from tests.helpers import unpack_batch

seq = W.seq
TEXT = text(140_000, 7)


def comp(lit, seqs=(), **kw):
    return dict(kind="comp", lit=lit, seqs=list(seqs), **kw)


def raw_lit(data, **kw):
    return dict(mode="raw", data=bytes(data), **kw)


def rle_lit(byte, n, **kw):
    return dict(mode="rle", data=bytes([byte]) * n, **kw)


def huf(data, **kw):
    return dict(mode="huf", data=bytes(data), **kw)


def treeless(data, **kw):
    return dict(mode="treeless", data=bytes(data), **kw)


def frame(*blocks, **kw):
    return dict(blocks=list(blocks), **kw)


# a sequence mix whose codes every table below covers: LL codes 0..20, OF codes 2..9, ML codes 0..24
def _mix(n, first_off=5):
    out = []
    for i in range(n):
        ll = (i * 7) % 21
        out.append(seq(ll, first_off + (i * 37) % 500, 3 + (i * 5) % 25) if i % 3 else (ll, 1 + i % 3, 3 + i % 20))
    return out


def _fse(log, used, rng=None, neg=(), extra=()):
    """normalized counts over `used` codes (plus `extra`), the codes in `neg` at "less than 1", the rest shared out"""
    size = 1 << log
    syms = sorted(set(used) | set(extra))
    norm = [0] * (max(syms) + 1)
    for s in syms:
        norm[s] = -1 if s in neg else 1
    pos = [s for s in syms if s not in neg]
    left = size - sum(1 for s in syms)
    for i in range(left):
        norm[pos[(i * 7 + (int(rng.integers(0, len(pos))) if rng is not None else 0)) % len(pos)]] += 1
    return ("fse", log, norm)


def _codes(seqs):
    return ({W.ll_code(s[0]) for s in seqs}, {W.highbit(s[1]) for s in seqs}, {W.ml_code(s[2]) for s in seqs})


def _tables_for(seqs, ll_log=6, of_log=5, ml_log=6, neg=True):
    llc, ofc, mlc = _codes(seqs)
    n = lambda c: {max(c)} if neg and len(c) > 1 else set()  # noqa: E731
    return dict(ll=_fse(ll_log, llc, neg=n(llc)), of=_fse(of_log, ofc, neg=n(ofc)), ml=_fse(ml_log, mlc, neg=n(mlc)))


def _lits(n, seed):
    return text(n, seed)


# ---------------------------------------------------------------------------------------------------------------------
# fillers put between the block that defines a table / tree and the block that re-uses it
FILLERS = {
    "raw_block": [dict(kind="raw", data=b"-raw block-")],
    "rle_block": [dict(kind="rle", byte=0x2A, size=77)],
    "noseq_raw_lits": [comp(raw_lit(b"raw literals, no sequences"))],
    "noseq_rle_lits": [comp(rle_lit(0x41, 40))],
    "all": [dict(kind="raw", data=b"r"), comp(rle_lit(0x42, 9)), dict(kind="rle", byte=1, size=3), comp(raw_lit(b"xyz"))],
}


HIST = dict(kind="raw", data=text(600, 11))  # history for the matches of _mix (no tables, no tree)


def _with_fillers(name, blocks, at, **kw):
    """the case, and the case with each filler inserted before block `at` (the user of what an earlier block defined);
    every one starts with HIST"""
    yield name, frame(HIST, *blocks, **kw)
    for fname, fill in FILLERS.items():
        yield f"{name}+{fname}", frame(HIST, *blocks[:at], *fill, *blocks[at:], **kw)


def valid_cases():
    """(name, description) of the named valid frames"""
    out = []
    add = out.append
    s1 = _mix(40)
    s2 = [(0, 1, 10), (4, 2, 5), (0, 3, 7)] + _mix(12, 9)
    lits1, lits2 = _lits(400, 1), _lits(300, 2)
    # Repeat_Mode re-using a Predefined, an RLE and an FSE table; across blocks without sequences
    out += _with_fillers("repeat_of_predefined", [comp(huf(lits1), s1), comp(raw_lit(lits2), s2, ll="rep", of="rep", ml="rep")], 1)
    rle_seqs = [seq(2, 17, 6)] * 5 + [(2, 1, 6)] * 20
    rle2 = [(1, 1, 6)] * 9 + [seq(1, 17, 6)]
    out += _with_fillers("repeat_of_rle", [comp(raw_lit(lits1[:100]), rle_seqs, ll=("rle", 2), of="pre", ml=("rle", 3)),
                                           comp(raw_lit(lits1[:60]), rle2, ll=("rle", 1), of="rep", ml="rep")], 1)
    out += _with_fillers("repeat_of_all_rle", [comp(raw_lit(lits1[:50]), [seq(2, 6, 4)] * 8, ll=("rle", 2), of=("rle", 3), ml=("rle", 1)),
                                               comp(raw_lit(lits1[:50]), [seq(2, 6, 4)] * 3, ll="rep", of="rep", ml="rep")], 1)
    t = _tables_for(s1 + s2)
    out += _with_fillers("repeat_of_fse", [comp(huf(lits1), s1, **t), comp(huf(lits2), s2, ll="rep", of="rep", ml="rep"),
                                           comp(treeless(lits2[:90]), _mix(5, 11), ll="rep", of="rep", ml="rep")], 1)
    mixed_t = dict(ll="rep", of=_fse(5, _codes(s2)[1]), ml="pre")
    out += _with_fillers("repeat_some_tables", [comp(raw_lit(lits1), s1, **t), comp(raw_lit(lits2), s2, **mixed_t),
                                                comp(raw_lit(lits2), s2, ll="rep", of="rep", ml="rep")], 1)
    # Treeless literals, tree defined two and more blocks back, over Raw / RLE literals
    big = _lits(5000, 3)
    out += _with_fillers("treeless_far_back", [comp(huf(big[:2000], streams=4), _mix(6)), comp(raw_lit(b"plain")), comp(rle_lit(0x61, 33)),
                                               comp(treeless(big[2000:2400]), _mix(4, 7)), comp(treeless(big[2400:4000], streams=4))], 1)
    out += _with_fillers("treeless_1_stream", [comp(huf(big[:200])), comp(treeless(big[200:700]))], 1)
    # "rep0 - 1" and the other repeat codes out of the previous block's history
    for name, s in (("rep0_minus_1", (0, 3, 9)), ("rep1_ll0", (0, 1, 9)), ("rep2_ll0", (0, 2, 9)), ("rep1", (3, 2, 9)), ("rep2", (3, 3, 9))):
        blocks = [comp(raw_lit(lits1[:200]), [seq(50, 40, 20), seq(30, 120, 11), seq(40, 9, 30)]), comp(raw_lit(lits2[:40]), [s, (2, 1, 4), s])]
        out += _with_fillers(name, blocks, 1)
    out.append(("rep0_minus_1_same_block", frame(comp(raw_lit(lits1[:20]), [seq(12, 9, 5), (0, 3, 5), (0, 3, 5), (4, 1, 6)]))))
    out.append(("rep_initial_history", frame(comp(raw_lit(lits1[:20]), [(9, 2, 5), (2, 3, 5), (0, 1, 6)]))))
    # FSE table descriptions at the edges
    s = _mix(60)
    llc, ofc, mlc = _codes(s)
    lits1 = _lits(1000, 4)
    add(("fse_log5", frame(HIST, comp(raw_lit(lits1), s, ll=_fse(5, llc), of=_fse(5, ofc), ml=_fse(5, mlc)))))
    add(("fse_max_log", frame(HIST, comp(raw_lit(lits1), s, ll=_fse(9, llc), of=_fse(8, ofc), ml=_fse(9, mlc)))))
    add(("fse_less_than_1", frame(HIST, comp(raw_lit(lits1), s, ll=_fse(6, llc, neg=set(list(llc)[::2])), of=_fse(5, ofc, neg=set(list(ofc)[1:])),
                                       ml=_fse(6, mlc, neg=set(list(mlc)[:-1]))))))
    # zero runs of 1, 2, 3, 4, 6, 3 and 14 symbols (the flags chain 3 + 3 + ... + the rest)
    gaps = dict(ll=("fse", 6, [20, 0, 11, 0, 0, 10, 0, 0, 0, 8, 0, 0, 0, 0, 5, 0, 0, 0, 0, 0, 0, 10]),
                of=("fse", 5, [0] * 14 + [10, 22]),
                ml=("fse", 6, [0] * 14 + [-1] + [0] * 3 + [63]))
    add(("fse_repeat_zero_flags", frame(dict(kind="raw", data=TEXT[:45_000]),
                                        comp(raw_lit(lits1), [seq(0, 20000, 17), seq(2, 40000, 21), seq(5, 17000, 17), seq(9, 33000, 21),
                                                              seq(14, 20000, 17), seq(28, 20000, 17)], **gaps), fcs=4)))
    # the last symbol takes the remainder; a symbol with the whole table (probability 1)
    add(("fse_last_takes_rest", frame(HIST, comp(raw_lit(lits1), s, ll=("fse", 6, [1] * 20 + [44]), of=("fse", 5, [1] * 9 + [23]),
                                           ml=("fse", 6, [1] * 24 + [-1, 39])))))
    add(("fse_whole_table", frame(HIST, comp(raw_lit(lits1[:100]), [seq(4, 20, 7)] * 9, ll=("fse", 5, [0, 0, 0, 0, 32]), of=("fse", 5, [0] * 4 + [32]),
                                       ml=("fse", 6, [0, 0, 0, 0, 64])))))
    # Huffman weights in both forms and at the length limit
    add(("huf_direct_odd", frame(comp(huf(b"abcabcabd" * 5, wform="direct")))))  # 'a'..'d' -> 100 weights, 99 written
    add(("huf_direct_even", frame(comp(huf(b"\x00\x01\x02\x00\x00\x05" * 9, wform="direct")))))
    add(("huf_fse_weights", frame(comp(huf(big[:3000], wform="fse", streams=4)))))
    add(("huf_fse_weights_log5", frame(HIST, comp(huf(big[:3000], wform="fse", wlog=5, streams=4), _mix(5)))))
    add(("huf_fse_weights_all_bytes", frame(comp(huf(rand(4000, 5) + bytes(range(256)), streams=4)))))
    w11 = [0] * 97 + [1, 1] + list(range(2, 11)) + [11]  # lengths 11, 11, 10, ..., 2, 1
    add(("huf_11_bit_codes", frame(comp(huf(bytes(range(97, 109)) * 3 + b"l" * 900, weights=w11, streams=4)))))
    add(("huf_11_bit_codes_fse", frame(comp(huf(bytes(range(97, 109)) * 3 + b"l" * 900, weights=w11, wform="fse")))))
    add(("huf_limit_6", frame(comp(huf(big[:4000], max_bits=6, streams=4)))))
    # four streams whose last segment is empty, and around it
    for n in (6, 7, 8, 9, 10, 13):
        add((f"huf4_regen_{n}", frame(comp(huf(b"abcdefghijklm"[:n], streams=4)))))
    # literals section header forms at their boundaries, minimal and forced
    for n in (0, 1, 31, 32, 4095, 4096):
        add((f"raw_lits_{n}", frame(comp(raw_lit(TEXT[:n])))))
        add((f"rle_lits_{n}", frame(comp(rle_lit(0x33, max(n, 1))))))
    add(("raw_lits_hdr3_forced", frame(comp(raw_lit(b"abc", hdr=3)))))
    add(("raw_lits_hdr2_forced", frame(comp(raw_lit(b"abc", hdr=2)))))
    add(("rle_lits_hdr3_forced", frame(comp(rle_lit(7, 5, hdr=3)))))
    add(("raw_lits_largest_block", frame(comp(raw_lit(TEXT[:131068])), fcs=4, single=False)))  # (a 131 072-byte block)
    for n in (1023, 1024, 16383, 16384, 100_000):
        add((f"huf4_lits_{n}", frame(comp(huf(TEXT[:n], streams=4)))))
    add(("huf1_lits_1023", frame(comp(huf(bytes(97 + b % 8 for b in TEXT[:1023]), max_bits=4)))))
    add(("huf4_hdr5_forced", frame(comp(huf(TEXT[:500], streams=4, hdr=5)))))
    add(("huf4_hdr4_forced", frame(comp(huf(TEXT[:500], streams=4, hdr=4)))))
    add(("huf4_hdr3_4streams", frame(comp(huf(TEXT[:500], streams=4, hdr=3)))))
    # Number_of_Sequences forms
    for n, form in ((127, None), (128, None), (5, 2), (0x7EFF, None), (0x7F00, None), (0x7F00 + 300, None)):
        seqs = [(0, 1, 3)] * n
        add((f"nseq_{n}_form{form or 'min'}", frame(HIST, comp(raw_lit(b"abc"), seqs, nseq_form=form, ll=("rle", 0), of=("rle", 0), ml=("rle", 0)))))
    # LL / ML codes at the top, a far offset across blocks, a block of exactly 128 KiB
    add(("ll35_ml52", frame(comp(raw_lit(TEXT[:70_000]), [seq(66_000, 4000, 600)]), comp(raw_lit(b"z"), [seq(1, 70_000, 66_000)]), fcs=4)))
    add(("far_offset", frame(dict(kind="raw", data=TEXT[:131_072]), dict(kind="raw", data=TEXT[5:100]),
                             comp(raw_lit(b"x"), [seq(1, 131_075, 200)]), single=False)))
    add(("block_128k_exact", frame(comp(raw_lit(TEXT[:1000]), [seq(1000, 700, 130_072)]), fcs=4)))
    # Frame_Content_Size of every width (the 2-byte field: value - 256), Dictionary_ID fields holding 0, no FCS
    for width, n in ((1, 0), (1, 255), (2, 256), (2, 65791), (4, 65792), (8, 300), (4, 0), (0, 500)):
        add((f"fcs_w{width}_{n}", frame(comp(raw_lit(TEXT[:n])), fcs=width, single=width != 0, window=0x30, checksum=n % 2 == 1)))
    for dw in (1, 2, 4):
        add((f"did_zero_w{dw}", frame(comp(huf(TEXT[:300])), did=(dw, 0), single=dw != 2)))
    # no Frame_Content_Size and two blocks: the one-shot call sizes its output at 128 KiB a block, the frame is shorter
    add(("no_fcs_multi_block", frame(dict(kind="raw", data=b"ab"), comp(huf(b"c")), single=False, fcs=0)))
    add(("no_fcs_multi_block_checksum", frame(HIST, comp(huf(TEXT[:3000], streams=4), _mix(9)), single=False, fcs=0, checksum=True)))
    add(("window_1k_small_blocks", frame(dict(kind="raw", data=TEXT[:1024]), comp(raw_lit(b"abc"), [seq(3, 1000, 500)]), single=False, window=0)))
    return out


def invalid_cases():
    """(name, description, status the decoder reports, why).  Each is one the reference's streaming decoder refuses;
    libzstd's error names are given where its code differs from the one reported (both are "corrupted" in kind)."""
    L = _lits(200, 9)
    w = W.weights_from_data(L)
    return [
        ("treeless_first", frame(comp(treeless(L, weights=w))), 20, "no earlier Huffman tree"),
        ("treeless_after_raw_lits", frame(comp(raw_lit(L)), comp(treeless(L, weights=w))), 20, "Raw literals leave no tree"),
        ("repeat_first", frame(comp(raw_lit(L), [seq(3, 5, 4)], ll=("rep", "pre"))), 20, "no earlier table"),
        ("repeat_after_noseq", frame(comp(huf(L)), comp(raw_lit(L), [seq(3, 5, 4)], ml=("rep", "pre"))), 20, "a block without sequences leaves no table"),
        ("lits_longer_than_section", frame(comp(raw_lit(L, size=300))), 20, "Regenerated_Size past the block"),
        ("seqs_use_more_lits", frame(comp(raw_lit(L[:10]), [seq(8, 3, 4), seq(8, 3, 4)])), 20, "literals run out"),
        ("offset_before_start", frame(comp(raw_lit(L[:10]), [seq(5, 6, 4)])), 20, "the match starts before the frame"),
        ("rep_offset_before_start", frame(comp(raw_lit(L[:10]), [(2, 3, 4)])), 20, "rep2 = 8 reaches before the frame"),
        ("block_over_128k", frame(comp(raw_lit(L[:1000]), [seq(1000, 700, 130_073)]), fcs=4), 20, "a block regenerates 128 KiB + 1"),
        ("nonzero_dictionary_id", frame(comp(raw_lit(L)), did=(1, 7)), 32, "libzstd: dictionary_wrong (32)"),
        ("ll_log_10", frame(comp(raw_lit(L), [seq(3, 5, 4)], ll=("fse", 10, [0, 0, 0, 1000, 24]))), 20, "LL accuracy log above 9"),
        ("of_log_9", frame(comp(raw_lit(L), [seq(3, 5, 4)], of=("fse", 9, [0, 0, 0, 500, 12]))), 20, "OF accuracy log above 8"),
        ("huf_12_bit_code", frame(comp(huf(b"ab" * 10 + b"c", weights=[0] * 97 + [11, 11, 12], wform="direct"))), 20, "a code length of 12"),
        ("seq_bits_left_over", frame(comp(raw_lit(L), _mix(10), extra_bits=3)), 20, "the bitstream is not consumed"),
        ("seq_bits_left_byte", frame(comp(raw_lit(L), _mix(10), extra_bits=8)), 20, "a whole byte is left"),
        ("seq_bits_overrun", frame(comp(raw_lit(L), _mix(10), extra_bits=-2)), 20, "the bitstream runs out"),
        ("huf4_regen_5", frame(comp(huf(b"abcde", streams=4))), 20, "four streams of 2, 2, 2, -1 bytes"),
        ("fcs_mismatch", frame(comp(raw_lit(L)), fcs_value=len(L) + 1, fcs=4), 20, "Frame_Content_Size differs"),
    ]


def window_cases():
    """Frames that break the window rule (block or offset beyond a 1 KiB window): the verdict is the reference's own
    (a streaming decoder holds more history than the window)."""
    return [
        ("block_over_window", frame(dict(kind="raw", data=TEXT[:2000]), single=False, window=0)),
        ("comp_block_over_window", frame(comp(raw_lit(TEXT[:1500])), single=False, window=0)),
        ("offset_over_window", frame(dict(kind="raw", data=TEXT[:1000]), dict(kind="raw", data=TEXT[1000:2000]), dict(kind="raw", data=TEXT[2000:3000]),
                                     comp(raw_lit(b"ab"), [seq(2, 2000, 10)]), single=False, window=0)),
    ]


# ---------------------------------------------------------------------------------------------------------------------
# random descriptions
def _random_norm(rng, used, max_sym, max_log):
    min_log = max(5, (len(used) - 1).bit_length())
    for _ in range(10):
        log = int(rng.integers(min_log, max_log + 1))
        size = 1 << log
        syms = set(used)
        for _ in range(int(rng.integers(0, 6))):
            syms.add(int(rng.integers(0, max_sym + 1)))
        if len(syms) > size:
            continue
        syms = sorted(syms)
        neg = {s for s in syms if rng.random() < 0.15}
        pos = [s for s in syms if s not in neg] or [syms[0]]
        neg -= set(pos)
        norm = [0] * (syms[-1] + 1)
        for s in syms:
            norm[s] = -1 if s in neg else 1
        left = size - len(syms)
        share = rng.multinomial(left, rng.dirichlet(np.ones(len(pos)) * 0.5)) if left else [0] * len(pos)
        for s, k in zip(pos, share):
            norm[s] += int(k)
        return ("fse", log, norm)
    return "pre"


def _pick_size(rng, cap):
    n = int(rng.choice([0, 1, 5, 6, 9, 10, 31, 32, 100, 1023, 1024, 4095, 4096, 16383, 16384, 30000])) + int(rng.integers(-1, 2))
    return max(0, min(n, cap))


def random_description(rng):
    """A valid random frame description: block mixes, literal modes, tables (Predefined, RLE, random normalized counts
    with "less than 1" entries and gaps, Repeat), repeat codes, sizes around header boundaries."""
    alpha = sorted(set(int(x) for x in rng.integers(0, int(rng.choice([4, 40, 256])), int(rng.integers(2, 60)))))
    if len(alpha) < 2:
        alpha.append((alpha[0] + 1) % 256)
    limit = max(int(rng.choice([11, 11, 9, 7])), (len(alpha) - 1).bit_length() + 1)
    src = bytes(int(x) for x in rng.choice(alpha, 200_000))
    blocks = []
    out_len = 0
    rep = [1, 4, 8]
    have_tree = False
    prev = {}
    for _ in range(int(rng.integers(1, 7))):
        kind = int(rng.integers(0, 10))
        if kind == 0:
            n = _pick_size(rng, 20_000)
            blocks.append(dict(kind="raw", data=bytes(rng.integers(0, 256, n, dtype=np.uint8))))
            out_len += n
            continue
        if kind == 1:
            n = _pick_size(rng, W.BLOCK_MAX)
            blocks.append(dict(kind="rle", byte=int(rng.integers(0, 256)), size=n))
            out_len += n
            continue
        nlit = _pick_size(rng, 40_000)
        lmode = rng.choice(["raw", "rle", "huf", "huf", "treeless"] if have_tree else ["raw", "rle", "huf"])
        if lmode in ("huf", "treeless") and nlit == 0:
            nlit = 1
        if lmode == "rle":
            nlit = max(nlit, 1)
        a = int(rng.integers(0, len(src) - nlit))
        data = src[a : a + nlit] if lmode != "rle" else bytes([int(rng.choice(alpha))]) * nlit
        if lmode == "raw" and rng.integers(0, 2):
            data = bytes(rng.integers(0, 256, nlit, dtype=np.uint8))
        lit = dict(mode=str(lmode), data=data)
        if lmode in ("huf", "treeless"):
            lit["streams"] = 4 if nlit > 1023 or (nlit >= 6 and rng.integers(0, 2)) else 1
        if lmode == "huf":
            weights = W.weights_from_data(data, int(rng.integers(limit, 12)), extra=alpha)
            lit["weights"] = weights
            forms = (["direct"] if len(weights) <= 129 else []) + (["fse"] if len(weights) >= 3 else [])
            lit["wform"] = str(rng.choice(forms))
            if lit["wform"] == "fse":
                lit["wlog"] = int(rng.choice([5, 6]))
                try:
                    W.weights_fse(weights, lit["wlog"])
                except AssertionError:
                    lit["wform"] = "direct"
                    if len(weights) > 129:
                        lit = dict(mode="raw", data=data)
            have_tree = have_tree or lit["mode"] == "huf"
        if lit["mode"] in ("raw", "rle") and rng.integers(0, 4) == 0:
            fits = [h for h, m in ((1, 31), (2, 4095), (3, 1 << 20)) if nlit <= m]
            lit["hdr"] = int(rng.choice(fits))
        # sequences
        nseq = int(rng.choice([0, 0, 1, 2, 5, 30, 200, 1000]))
        seqs = []
        lits_left = nlit
        room = W.BLOCK_MAX - nlit
        for _ in range(nseq):
            ll = int(rng.integers(0, min(lits_left, int(rng.choice([3, 20, 300]))) + 1))
            ml = int(rng.choice([3, 4, int(rng.integers(3, 40)), int(rng.integers(3, 600)), int(rng.integers(3, 5000))]))
            if ml > room:
                break
            pos = out_len + ll
            r = int(rng.integers(0, 4))
            ov = None
            if r < 3:
                try:
                    off, _ = W.resolve(rep, ll, r + 1)
                    if off <= pos:
                        ov = r + 1
                except ValueError:
                    pass
            if ov is None:
                if pos == 0:
                    break
                far = int(rng.choice([1, 8, 100, 5000, 70_000, 140_000]))
                ov = min(pos, int(rng.integers(1, far + 1))) + 3
            _, rep = W.resolve(rep, ll, ov)
            seqs.append((ll, ov, ml))
            lits_left -= ll
            room -= ml
            out_len += ll + ml
        out_len += lits_left
        b = comp(lit, seqs)
        if seqs:
            for kind, codes, max_sym in (("ll", [W.ll_code(s[0]) for s in seqs], 35), ("of", [W.highbit(s[1]) for s in seqs], 31),
                                         ("ml", [W.ml_code(s[2]) for s in seqs], 52)):
                choice = int(rng.integers(0, 5))
                t = prev.get(kind)
                if choice == 0 and t is not None and set(codes) <= set(t.by_sym):
                    b[kind] = "rep"
                    continue
                if choice == 1 and len(set(codes)) == 1:
                    spec = ("rle", codes[0])
                elif choice <= 2 and max(codes) <= (28 if kind == "of" else max_sym):
                    spec = "pre"
                else:
                    spec = _random_norm(rng, sorted(set(codes)), max_sym, W.MAX_LOG[kind])
                    if spec == "pre" and max(codes) > 28 and kind == "of":
                        spec = _random_norm(rng, sorted(set(codes)), max_sym, W.MAX_LOG[kind])
                b[kind] = spec
                prev[kind] = W._table(kind, spec, None)[2]
            nmin = 1 if len(seqs) < 128 else 2 if len(seqs) < 0x7F00 else 3
            if nmin < 3 and rng.integers(0, 4) == 0:
                b["nseq_form"] = 2
        blocks.append(b)
    single = bool(rng.integers(0, 2))
    d = dict(blocks=blocks, single=single, checksum=bool(rng.integers(0, 2)), did=(int(rng.choice([0, 0, 1, 2, 4])), 0))
    if not single:
        d["window"] = int(rng.choice([0x58, 0x80, 0x41]))
    if rng.integers(0, 3) == 0:
        widths = [0] if not single else [1] if out_len <= 255 else []
        widths += ([2] if 256 <= out_len <= 65791 else []) + ([4] if out_len < 1 << 32 else []) + [8]
        d["fcs"] = int(rng.choice(widths))
    return d


# ---------------------------------------------------------------------------------------------------------------------
def check_writer(cases):
    """Every valid description: libzstd one-shot, the reference's streaming call sequence and the C oracle restore
    exactly execute(description).  Returns the C oracle's statistics summed over the frames."""
    tot = {}
    for name, d in cases:
        f = W.write(d)
        exp = W.execute(d)
        assert ref_path.ref_decompress(f, len(exp) + 64) == exp, (name, "libzstd one-shot")
        assert ref_path.ref_decompress_stream(f + b"\x28\xb5\x2f\xfdnext", 0) == exp, (name, "libzstd streaming")
        got, err, used, st = ref_path.c_zstd_decompress_frame(f, len(exp) + 64)
        assert err == 0 and got == exp and used == len(f), (name, "C oracle", err)
        for k, v in st.items():
            tot[k] = tot.get(k, 0) + v
    return tot


def _ref_rejects(f):
    try:
        ref_path.ref_decompress_stream(f + b"\x28\xb5\x2f\xfdnext", 0)
        return False
    except ref_path.ZstdError:
        return True


# the decode paths: (name, split_min, chain mode, chunk blocks).  split_min 2^40 keeps every frame on the lane-per-frame
# decoder (multi-block frames walked serially); 1 stages every frame of two blocks and more.
PATHS = [("lane", 1 << 40, 1, 0), ("staged_chain0", 1, 0, 0), ("staged_chain2", 1, 2, 0), ("staged_chunk1", 1, 1, 1)]


def _set_path(lib, split_min, chain, chunk):
    lib.dll.zg_internal_set_decode_split_min(C.c_uint64(split_min))
    lib.dll.zg_internal_set_decode_chain_mode(C.c_uint32(chain))
    lib.dll.zg_internal_set_decode_chunk_blocks(C.c_uint32(chunk))


def _b3(d):
    return ref_path.c_blake3(d)


def _one_shot(lib, d, f, cap):
    dst = C.create_string_buffer(max(cap, 1))
    r = lib.zg_decompress(d, dst, cap, f, len(f))
    if lib.zg_is_error(r):
        return None, lib.zg_get_error_code(r)
    return dst.raw[:r], 0


def run_frames(lib, items, rng, alone=True):
    """items: (name, frame, expected bytes or None, expected status, size the caller claims).  Every path, each frame alone and all of them in
    one batch (a warp decodes up to 32 frames side by side), then the one-shot and the streaming entry points."""
    from tests.fuzz_cases import _stream_once

    ulens = [ul for *_, ul in items]
    digs = [_b3(e if e is not None else b"") for _, _, e, _, _ in items]
    want_st = [st for _, _, _, st, _ in items]
    try:
        for pname, *cfg in PATHS:
            _set_path(lib, *cfg)
            groups = [[i] for i in range(len(items))] if alone else []
            order = list(range(len(items)))
            rng.shuffle(order)
            step = 12 if cfg[2] == 1 else len(order)  # (a chunk of one block per launch is slow on the emulator)
            groups += [order[i : i + step] for i in range(0, len(order), step)]
            for g in groups:
                outs, ok, status, rc = unpack_batch(lib, [items[i][1] for i in g], [ulens[i] for i in g], [digs[i] for i in g])
                for j, i in enumerate(g):
                    name, _, exp, st, _ = items[i]
                    assert status[j] == st, (pname, name, "status", status[j], st)
                    if exp is not None:
                        assert outs[j] == exp and ok[j] == 1, (pname, name, "bytes differ from the description's")
                    else:
                        assert ok[j] == 0, (pname, name)
                bad = [want_st[i] for i in g if want_st[i]]
                if bad:
                    assert lib.zg_is_error(rc) and lib.zg_get_error_code(rc) == bad[0], (pname, "return code", rc)
                else:
                    assert rc == 0, (pname, rc)
    finally:
        _set_path(lib, 0, 1, 0)
    d = lib.zg_dctx_create()
    try:
        for name, f, exp, st, ul in items:
            got, err = _one_shot(lib, d, f, ul + 64)
            assert err == st and (exp is None or got == exp), (name, "zg_decompress", err, st)
            got, _used, err = _stream_once(lib, d, f + b"\x28\xb5\x2f\xfdnext", rng, 1 << 30)
            if exp is not None:
                assert err == 0 and got == exp, (name, "zg_decompress_stream", err)
            else:
                assert err != 0, (name, "zg_decompress_stream accepted an invalid frame")
                if err == -1:
                    lib.zg_dctx_free(d)
                    d = lib.zg_dctx_create()
    finally:
        lib.zg_dctx_free(d)


def _items_valid(cases):
    out = []
    for name, d in cases:
        exp = W.execute(d)
        out.append((name, W.write(d), exp, 0, len(exp)))
    return out


def handmade_frames(lib, first, count, log=None, named=True):
    """The named valid and invalid frames (when `named`) and `count` random descriptions from seed `first`, through every
    decode path of `lib`.  Returns {"valid": frames restored, "invalid": frames rejected}."""
    rng = np.random.default_rng(first)
    n_valid = n_invalid = 0
    if named:
        items = _items_valid(valid_cases())
        bad = []
        for name, d, st, _why in invalid_cases():
            f = W.write(d)
            assert _ref_rejects(f), (name, "the reference accepts this frame")
            bad.append((name, f, None, st, W.nominal_size(d)))
        for name, d in window_cases():
            f = W.write(d)
            if _ref_rejects(f):
                bad.append((name, f, None, 20, W.nominal_size(d)))
            else:
                items.append((name, f, W.execute(d), 0, W.nominal_size(d)))
        run_frames(lib, items + bad, rng)
        n_valid += len(items)
        n_invalid += len(bad)
    for seed in range(first, first + count):
        r = np.random.default_rng(seed)
        cases = [(f"seed{seed}.{i}", random_description(r)) for i in range(8)]
        check_writer(cases)
        run_frames(lib, _items_valid(cases), r, alone=False)
        n_valid += len(cases)
        if log:
            log(seed, n_valid)
    return dict(valid=n_valid, invalid=n_invalid)

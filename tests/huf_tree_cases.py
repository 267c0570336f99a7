"""Single-block frames whose Huffman literals the decoder reads ahead of the fused kernel (k_zd_huf_literals, one lane
per tree), with tree descriptions, jump tables and streams at every edge it checks.  They run in batches of more than
32 frames, good and bad shuffled together, so that a bad tree shares a warp's group of sections with good ones.  Every
verdict is checked three ways: against the case's expected verdict, against libzstd, and against the same literals in
a two-block frame, which is not decoded ahead: the warp that decodes its block reads the tree there, on whichever path
takes the frame.  Shared by tests/test_huf_trees_emu.py and tests/test_huf_trees_gpu.py."""
import struct

import numpy as np

from oracle import ref_path
from tests import zstd_writer as W
from tests.golden.recipes import rand, text
from tests.helpers import unpack_batch

CORRUPT = 20


def frame(section, regen, lead_block=False):
    """A frame of one compressed block (literals `section`, no sequences) that regenerates `regen` bytes.  With
    `lead_block` an empty Raw block comes first, so that the frame is a multi-block one."""
    body = section + b"\0"
    out = bytearray(struct.pack("<I", 0xFD2FB528))
    if regen < 256:
        out += bytes([0x20, regen])
    elif regen < 65536 + 256:
        out += bytes([0x60]) + struct.pack("<H", regen - 256)
    else:
        out += bytes([0xA0]) + struct.pack("<I", regen)
    if lead_block:
        out += bytes(3)
    out += struct.pack("<I", 1 | 2 << 1 | len(body) << 3)[:3] + body
    return bytes(out)


def direct_tree(explicit):
    """A direct tree description of the explicit weights, whatever they are"""
    ex = list(explicit) + [0] * (len(explicit) & 1)
    return bytes([127 + len(explicit)]) + bytes((ex[i] << 4) | ex[i + 1] for i in range(0, len(ex), 2))


def fse_tree(weights, norm, log=6):
    """W.weights_fse with the normalised counts given: they may declare symbols the weights never use"""
    ex = list(weights[:-1])
    t = W.FseTable(log, norm)
    m = len(ex)
    a, b = ex[0::2], ex[1::2]
    pen = a if (m - 2) % 2 == 0 else b
    last_state = next(i for i in t.by_sym[pen[-1]] if t.states[i][1] > 0)
    chains = []
    for c in (a, b):
        states = [last_state if c is pen else t.by_sym[c[-1]][0]]
        upd = []
        for s in reversed(c[:-1]):
            i, bits = t.prev_state(s, states[-1])
            upd.append((bits, t.states[i][1]))
            states.append(i)
        states.reverse()
        upd.reverse()
        chains.append((states, upd))
    fields = [(chains[0][0][0], log), (chains[1][0][0], log)]
    for j in range(m - 2):
        fields.append(chains[j % 2][1][j // 2])
    body = W.ncount_bytes(log, norm) + W.backward_stream(fields)
    assert len(body) < 128
    return bytes([len(body)]) + body


def section(data, weights=None, tree=None, streams=4, jump=None, regen=None):
    """(literals section, Regenerated_Size): `data` Huffman-coded with `weights` (from the data by default) under the
    tree description `tree` (direct or FSE as the writer picks), `jump` in place of the jump table, `regen` in place of
    the data's size"""
    weights = weights or W.weights_from_data(data)
    code = W.HufCode(weights)
    if tree is None:
        tree = W.weights_direct(weights) if len(weights) - 1 <= 128 else W.weights_fse(weights)
    if streams == 1:
        body = tree + code.stream(data)
    else:
        seg = (len(data) + 3) // 4
        parts = [code.stream(data[i * seg : (i + 1) * seg] if i < 3 else data[3 * seg :]) for i in range(4)]
        body = tree + (jump if jump is not None else struct.pack("<HHH", *(len(p) for p in parts[:3]))) + b"".join(parts)
    regen = len(data) if regen is None else regen
    return W.lit_header(2, regen, len(body), streams, 3 if streams == 1 else None) + body, regen


def _geometric(n, seed):
    """bytes with a long-tailed histogram: the longest codes reach the 11-bit limit"""
    rng = np.random.default_rng(seed)
    return bytes((np.minimum(rng.geometric(0.35, n), 200) + 30).astype(np.uint8))


def good_cases():
    """(name, section, regen) of valid sections"""
    out = []
    for i, n in enumerate((300, 700, 1306, 2500, 4049, 9000)):
        d = text(n, 11 + i)
        out.append((f"text{n}_direct", *section(d)))
        out.append((f"text{n}_fse", *section(d, tree=W.weights_fse(W.weights_from_data(d)))))
    for n in (40, 200, 900):
        d = text(n, 3)
        out.append((f"text{n}_1stream", *section(d, streams=1)))
        out.append((f"text{n}_1stream_fse", *section(d, streams=1, tree=W.weights_fse(W.weights_from_data(d)))))
    r = rand(6000, 5) + bytes(range(256))
    out.append(("all_256_symbols", *section(r)))  # 255 explicit weights, FSE-coded
    out.append(("two_symbols", *section(bytes([65, 66, 66, 65] * 50))))  # maxbits 1
    out.append(("two_symbols_1stream", *section(bytes([7, 9, 9]) * 20, streams=1)))
    g = _geometric(8000, 2)
    assert max(W.HufCode(W.weights_from_data(g)).code[s][1] for s in set(g)) == 11
    out.append(("maxbits11", *section(g)))
    out.append(("maxbits11_fse", *section(g, tree=W.weights_fse(W.weights_from_data(g)))))
    return out


def lenient_cases():
    """(name, section, regen, data) of sections the decoder accepts and libzstd rejects: FSE tables that declare weights above
    11 the stream never decodes.  The decoder reads a table's counts for up to 256 symbols and only rejects a weight it
    decodes; libzstd sizes its workspace for weights 0..11 and rejects the table."""
    out = []
    d = text(1500, 9)
    wts = W.weights_from_data(d)
    counts = [0] * 12
    for x in wts[:-1]:
        counts[x] += 1
    norm = W.normalize(counts, 6)
    norm[max(range(12), key=lambda k: norm[k])] -= 2
    norm += [0] * (201 - len(norm))
    norm[13], norm[200] = -1, 1
    out.append(("declares_unused_weights_13_200", *section(d, tree=fse_tree(wts, norm)), d))
    norm = W.normalize(counts, 6) + [1]
    norm[max(range(12), key=lambda k: norm[k])] -= 1
    out.append(("declares_unused_weight_12", *section(d, tree=fse_tree(wts, norm)), d))
    return out


def ncount_symbols(tree):
    """how many symbols the NCount of an FSE-coded tree description declares (RFC 8878 4.1.1), or 0 when unreadable"""
    bits = int.from_bytes(tree[1 : 1 + tree[0]], "little")
    n, pos = tree[0] * 8, 4
    remaining, sym = 1 << ((bits & 15) + 5), 0
    while remaining > 0 and sym <= 255 and pos <= n:
        nb = (remaining + 1).bit_length()
        thr = (1 << nb) - 1 - (remaining + 1)
        val = bits >> pos & ((1 << (nb - 1)) - 1)
        pos += nb - 1
        if val >= thr:
            hi = bits >> pos & 1
            pos += 1
            val = val | hi << (nb - 1)
            val -= thr if hi else 0
        sym += 1
        remaining -= 1 if val == 0 else val - 1
        if val == 1:
            while True:
                rep = bits >> pos & 3
                pos += 2
                sym += rep
                if rep != 3:
                    break
    return sym if pos <= n else 0


def bad_cases():
    """(name, section, regen) of sections the decoder must reject as corrupt"""
    out = []
    d = text(1200, 21)
    wts = W.weights_from_data(d)
    fse = W.weights_fse(wts)
    filler = b"\x5a" * 40 + b"\x81"

    def bad_tree(name, tree, streams=1):
        out.append((name, W.lit_header(2, 64, len(tree + filler), streams, 3) + tree + filler, 64))

    bad_tree("direct_weights_past_section", direct_tree([1] * 120)[:20])
    bad_tree("fse_csz_0", bytes([0]) + fse[1:])
    bad_tree("fse_csz_1", bytes([1]) + fse[1:])
    bad_tree("ncount_log_above_6", bytes([fse[0], fse[1] | 0x0F]) + fse[2:])
    nc = len(W.ncount_bytes(6, W.normalize([wts[:-1].count(k) for k in range(12)], 6)))
    bad_tree("ncount_truncated", bytes([2]) + fse[1:3] + fse[3:])
    bad_tree("ncount_fills_description", bytes([nc]) + fse[1 : 1 + nc] + fse[1 + nc :])
    bad_tree("weights_stream_no_marker", fse[:-1] + b"\0")
    many = [1, 2] * 150 + [1]
    bad_tree("more_than_254_weights", W.weights_fse(many))
    bad_tree("weight_above_11", direct_tree([12, 1, 1]))
    w12 = [12, 1, 1, 2, 1, 3, 1]
    bad_tree("weight_12_fse_coded", fse_tree(w12, W.normalize([w12[:-1].count(k) for k in range(13)], 6)))
    bad_tree("zero_sum", direct_tree([0, 0, 0]))
    bad_tree("maxbits_above_11", direct_tree([11, 11]))
    bad_tree("remainder_not_power_of_two", direct_tree([3, 1]))
    bad_tree("fewer_than_two_weights_of_1", direct_tree([2, 2]))
    # jump tables and streams
    tree = W.weights_direct(wts)
    t4 = W.lit_header(2, len(d), len(tree) + 9, 4, 3)
    out.append(("jump_table_under_10_bytes", t4 + tree + b"\x01\x00\x01\x00\x01\x00\x01\x01\x01", len(d)))
    sec, _ = section(d)
    avail = len(sec) - 3 - len(tree) - 6
    out.append(("jump_sizes_fill_section", *section(d, jump=struct.pack("<HHH", avail - 2, 1, 1))))
    out.append(("jump_sizes_past_section", *section(d, jump=struct.pack("<HHH", avail, 0, 0))))
    out.append(("first_stream_empty", *section(d, jump=struct.pack("<HHH", 0, 40, 40))))
    for n in (1, 2, 5):  # 4 segments of (n + 3) / 4 do not fit n
        out.append((f"four_streams_of_{n}", *section(bytes([1, 2, 3, 4, 5])[:n])))
    s1, _ = section(d[:900], streams=1)
    out.append(("stream_marker_missing", s1[:-1] + b"\0", 900))
    out.append(("stream_one_symbol_short", *section(d[:900], streams=1, regen=899)))
    out.append(("stream_one_symbol_long", *section(d[:900], streams=1, regen=901)))
    return out


def ref_verdict(f):
    """libzstd's streaming decoder on the frame: its bytes, or None when it rejects the frame"""
    try:
        return ref_path.ref_decompress_stream(f + b"\x28\xb5\x2f\xfdnext", 0)
    except ref_path.ZstdError:
        return None


def decode(lib, frames, ulens, want):
    """single-block and two-block frames in one batch each: their statuses and outputs (digests from `want`)"""
    digs = [ref_path.c_blake3(w if w is not None else b"") for w in want]
    one = unpack_batch(lib, [frame(s, r) for s, r in frames], ulens, digs)
    two = unpack_batch(lib, [frame(s, r, lead_block=True) for s, r in frames], ulens, digs)
    return one, two


def check_cases(lib, seed):
    """every case, shuffled into one batch of more than 32.  Returns (good, bad) counts."""
    good, bad = good_cases(), bad_cases()
    lenient = {n: d for n, _, _, d in lenient_cases()}
    items = [(n, s, r, True) for n, s, r in good] + [(n, s, r, False) for n, s, r in bad]
    items += [(n, s, r, True) for n, s, r, _ in lenient_cases()]
    items += [(f"{n}#2", s, r, True) for n, s, r in good]  # a second copy, so that no group is mostly bad
    order = list(range(len(items)))
    np.random.default_rng(seed).shuffle(order)
    items = [items[i] for i in order]
    assert len(items) > 64
    want = []
    for name, s, r, ok in items:
        got = ref_verdict(frame(s, r))
        if name in lenient:
            assert got is None, (name, "libzstd accepts this table")
            got = lenient[name]
        else:
            assert (got is not None) == ok, (name, "libzstd's verdict differs from the case's")
        want.append(got)
    (outs, oks, st, _), (outs2, oks2, st2, _) = decode(lib, [(s, r) for _, s, r, _ in items], [r for _, _, r, _ in items], want)
    for j, (name, _, _, ok) in enumerate(items):
        if ok:
            assert st[j] == 0 and oks[j] == 1 and outs[j] == want[j], (name, st[j])
        else:
            assert st[j] == CORRUPT and oks[j] == 0, (name, st[j])
        assert (st2[j], oks2[j]) == (st[j], oks[j]), (name, "the two-block frame's verdict differs", st2[j], st[j])
    return len(good), len(bad)


def mutate_trees(lib, seed, rounds, per_round=48):
    """Random byte changes inside the tree descriptions of good sections.  Whatever the decoder accepts must equal what
    libzstd restores (but for the tables lenient_cases shows), and the single-block verdict must equal the two-block
    one.  Returns (accepted, rejected)."""
    rng = np.random.default_rng(seed)
    bases = []
    for i, n in enumerate((400, 1306, 3000)):
        d = text(n, 40 + i)
        wts = W.weights_from_data(d)
        for tree in (W.weights_direct(wts), W.weights_fse(wts)):
            sec, r = section(d, tree=tree, streams=1 if n < 1000 else 4)
            bases.append((sec, r, 3, len(tree)))  # (the 3-byte literals header comes first)
    sec, r = section(rand(3000, 8) + bytes(range(256)))
    bases.append((sec, r, 4, sec[4] + 1))
    acc = rej = 0
    for _ in range(rounds):
        frames, want, ats = [], [], []
        for _ in range(per_round):
            sec, r, at, tl = bases[int(rng.integers(len(bases)))]
            b = bytearray(sec)
            for _ in range(int(rng.integers(1, 4))):
                b[at + int(rng.integers(tl))] ^= int(rng.integers(1, 256))
            frames.append((bytes(b), r))
            ats.append(at)
            want.append(ref_verdict(frame(bytes(b), r)))
        (outs, oks, st, _), (outs2, oks2, st2, _) = decode(lib, frames, [r for _, r in frames], want)
        for j in range(per_round):
            assert st[j] in (0, CORRUPT), st[j]
            if st[j] == 0 and want[j] is None:
                tree = frames[j][0][ats[j] :]
                assert tree[0] < 128 and ncount_symbols(tree) > 12, ("accepted, but libzstd rejects it", frames[j])
                assert outs2[j] == outs[j]
                acc += 1
            elif st[j] == 0:
                assert outs[j] == want[j] and oks[j] == 1, ("accepted, but libzstd restores otherwise", frames[j])
                acc += 1
            else:
                rej += 1
            assert (st2[j], oks2[j]) == (st[j], oks[j]), ("the two-block frame's verdict differs", frames[j], st[j], st2[j])
    return acc, rej

"""Encoder conformance: inputs built to push this library's encoder onto one edge of the format each -- literals
section types and header sizes, Huffman length limit and weight descriptions, Number_of_Sequences header sizes,
sequence table modes, the longest literal runs and matches, the distance limit, block and frame header layout --
and the C oracle's statistics (oracle/zarc_oracle.c) asserting that the frame really took that edge.  Every frame is
also restored by libzstd (one-shot and the reference's streaming call sequence), by the C oracle and by this library's
decoder (digests verified), and every frame of more than one block is checked to be made of independent blocks: no
match reaches into an earlier block and no repeat code resolves to an offset set in one.

The match finder removes bytes, so the literal and sequence counts of a frame are not the input's size.  Inputs are
built from bytes it cannot match (`unique`: no 4-gram occurs twice) with the repeats put in on purpose, and every edge
is asserted on the statistics, never on the input.

Shared by the CPU test-suite (tests/test_encoder_edges_emu.py), the GPU suite (tests/test_encoder_edges_gpu.py) and the
rare-path builds there.  `run_cases` raises AssertionError naming the case and the edge it no longer reaches."""
import numpy as np

from oracle import ref_path
from oracle.ref_path import NONE_SEEN, lit_header_bytes
from tests.golden.recipes import text
from tests.helpers import pack_batch, unpack_batch

BLOCK = 131072
LEVELS = (1, 3, 9)


# ---------------------------------------------------------------------------------------------------------------------
# inputs
def unique(n, seed, alphabet=256, weights=None, seen=None):
    """n bytes drawn from `alphabet` symbols (optionally weighted) such that no 4-gram occurs twice, in this string or
    in `seen` (a set of 4-grams shared between the parts of one input).  Where no unseen 4-gram is left after a few
    draws the byte is taken anyway: callers assert the edge on the statistics."""
    rng = np.random.default_rng(seed)
    seen = set() if seen is None else seen
    p = None if weights is None else np.asarray(weights, float) / np.sum(weights)
    draws = rng.choice(alphabet, size=(n, 8), p=p)
    out = bytearray()
    for i in range(n):
        for c in draws[i]:
            g = bytes(out[-3:]) + bytes([c]) if i >= 3 else None
            if g is None or g not in seen:
                break
        out.append(int(c))
        if i >= 3:
            seen.add(bytes(out[-4:]))
    return bytes(out)


def skewed(n, seed, nsym=64, q=0.9, base=0):
    """unmatchable literals over symbols base.. base+nsym-1, weights q^k: Huffman pays"""
    return bytes((b + base) & 0xFF for b in unique(n, seed, nsym, q ** np.arange(nsym)))


def fib_weights(nsym):
    w = [1, 1]
    while len(w) < nsym:
        w.append(w[-1] + w[-2])
    return w


def with_sequences(k, seed, lit=(8, 12), ml=(5, 9), new_offsets=False, first=None):
    """k sequences: fresh bytes (a length in range(*lit)) and then a copy of the start of the fresh bytes before them (a
    length in range(*ml)).  Every fresh run is copied once and only by the next sequence: each copy is one match, found
    a few dozen bytes back, and nothing else repeats.  new_offsets: each offset differs from the three before it (no
    repeat codes) where the lengths leave a choice.  first: length of the run the first sequence copies from"""
    rng = np.random.default_rng(seed)
    seen = set()
    prev = unique(first or int(rng.integers(*lit)), seed, seen=seen)
    out = bytearray(prev)
    copied, offs, src = 0, [], b""  # length and source of the last copy; the offsets so far
    for j in range(k):
        n = int(rng.integers(*lit))
        if new_offsets:  # offset = this fresh run + the last copy + the fresh run before it
            n = int(rng.choice([x for x in range(*lit) if x + copied + len(prev) not in offs[-3:]] or [n]))
        offs.append(n + copied + len(prev))
        after = src[copied] if copied < len(src) else None  # the byte after the last copy's source
        before = out[len(out) - copied - len(prev) - 1] if len(out) > copied + len(prev) else None  # the byte before prev
        for t in range(100):  # neither copy may grow by a byte that happens to repeat its source's neighbour
            fresh = unique(n, seed * 100_000 + j + t * 7919, seen=set(seen))
            if fresh[0] != after and fresh[-1] != before:
                break
        seen.update(fresh[i : i + 4] for i in range(len(fresh) - 3))
        copied = int(rng.integers(*ml))
        out += fresh + prev[:copied]
        src, prev = prev, fresh
    return bytes(out)


def equal_weights(c=8, seed=0):
    """224 symbols c times each and symbol 224 32c times, no 4-gram twice: Huffman gives the 224 one weight and symbol 224
    (maxsym, whose weight is implied) another"""
    rng = np.random.default_rng(seed)
    while True:
        small = rng.permutation(np.repeat(np.arange(224, dtype=np.uint8), c))
        out = np.insert(small, np.arange(7, len(small) + 1, 7), 224).tobytes()
        if len({out[i : i + 4] for i in range(len(out) - 3)}) == len(out) - 3:
            return out


def exact_unique(counts, seed):
    """a string with exactly counts[s] bytes of value s and no 4-gram twice (a shuffle, each byte drawn so that its
    4-gram is new; drawn again from another seed if that gets stuck)"""
    rng = np.random.default_rng(seed)
    while True:
        pool = list(np.repeat(np.arange(len(counts)), counts))
        rng.shuffle(pool)
        out, seen = bytearray(), set()
        while pool:
            for t in range(min(len(pool), 64)):
                j = len(pool) - 1 - t
                g = bytes(out[-3:]) + bytes([pool[j]]) if len(out) >= 3 else None
                if g is None or g not in seen:
                    break
            else:
                break
            pool[j], pool[-1] = pool[-1], pool[j]
            out.append(int(pool.pop()))
            if g:
                seen.add(g)
        if not pool:
            return bytes(out)


def grams_walk(k=4, seed=0, n=BLOCK):
    """k 4-byte grams (distinct first bytes, distinct last bytes, every 4-gram across two grams distinct), then a walk
    over them in which no gram is followed by the gram that followed it last time: every gram is a match of exactly
    4 bytes at its previous occurrence, with no literal in between"""
    rng = np.random.default_rng(seed)
    while True:
        g = rng.integers(0, 256, (k, 4), dtype=np.uint8)
        g[:, 0], g[:, 3] = rng.permutation(256)[:k], rng.permutation(256)[:k]
        grams = [bytes(x) for x in g]
        if len(set(grams) | {(a + b)[i : i + 4] for a in grams for b in grams if a != b for i in (1, 2, 3)}) == k + 3 * k * (k - 1):
            break
    out, last, cur = bytearray(b"".join(grams)), {i: (i + 1) % k for i in range(k)}, k - 1
    while len(out) < n:
        s = (last[cur] + 1) % k
        s = (s + 1) % k if s == cur else s
        last[cur] = cur = s
        out += grams[s]
    return bytes(out[:n])


def huf_floor_raises(data, maxlog=11):
    """How often ze_huf_build raises its count floor on the histogram of `data` before the tree is at most `maxlog`
    deep: the same construction (floor total >> maxlog, doubled per retry; leaves sorted by (count, symbol); the two-queue
    merge taking the leaf on ties), restated plainly"""
    cnt = np.bincount(np.frombuffer(data, np.uint8), minlength=256)
    leaves = sorted((int(c), s) for s, c in enumerate(cnt) if c)
    n = len(leaves)
    limit = max(1, sum(c for c, _ in leaves) >> maxlog)
    for raises in range(32):
        nc = [max(c, limit) for c, _ in leaves] + [0] * (n - 1)
        par, q1, q2 = [0] * (2 * n - 1), 0, n
        for nn in range(n, 2 * n - 1):
            pair = []
            for _ in range(2):
                if q1 < n and (q2 >= nn or nc[q1] <= nc[q2]):
                    pair.append(q1)
                    q1 += 1
                else:
                    pair.append(q2)
                    q2 += 1
            nc[nn] = nc[pair[0]] + nc[pair[1]]
            par[pair[0]] = par[pair[1]] = nn
        depth = [0] * (2 * n - 1)
        for i in range(2 * n - 3, -1, -1):
            depth[i] = depth[par[i]] + 1
        if max(depth[:n]) <= maxlog:
            return raises
        limit <<= 1


def run_then_match(nlit, seed, back=64, ml=64):
    """nlit unmatchable bytes, then a copy of `ml` bytes from `back` bytes before the end of the run"""
    r = unique(nlit, seed)
    src = bytes(r[len(r) - back :][:ml])
    return r + src


# ---------------------------------------------------------------------------------------------------------------------
# checking
def pack_frames(lib, datas, level, params=()):
    """this library's encoder (zg_pack_batch, checksums on): one frame per input"""
    cctx = lib.zg_cctx_create()
    try:
        lib.check(lib.zg_cctx_init(cctx, 0))
        lib.check(lib.zg_cctx_set_parameter(cctx, 201, 1))
        lib.check(lib.zg_cctx_set_parameter(cctx, 100, level))
        for p, v in params:
            lib.check(lib.zg_cctx_set_parameter(cctx, p, v))
        lib.check(lib.zg_cctx_reset_archive(cctx, 12))
        r = pack_batch(lib, cctx, datas)
    finally:
        lib.zg_cctx_free(cctx)
    assert r["rc"] == 0, r["rc"]
    return [bytes(r["frames"][o - 12 : o - 12 + ln]) for o, ln in zip(r["off"], r["len"])]


def check_frames(lib, datas, frames, what=""):
    """every decoder restores every frame; returns the C oracle's statistics per frame"""
    stats = []
    for i, (d, fr) in enumerate(zip(datas, frames)):
        tag = (what, i, len(d))
        assert ref_path.ref_decompress(fr, len(d)) == d, (*tag, "libzstd one-shot")
        assert ref_path.ref_decompress_stream(b"\x01" * 3 + fr + b"tail", 3) == d, (*tag, "libzstd streaming")
        got, err, consumed, st = ref_path.c_zstd_decompress_frame(fr, len(d))
        assert err == 0 and got == d and consumed == len(fr), (*tag, "C oracle", err)
        if st["blocks"] > 1:
            assert st["xblock_matches"] == 0 and st["xblock_reps"] == 0, (*tag, "a block depends on an earlier one", st["xblock_matches"], st["xblock_reps"])
        stats.append(st)
    outs, ok, status, rc = unpack_batch(lib, frames, [len(d) for d in datas], [ref_path.c_blake3(d) for d in datas])
    assert rc == 0 and outs == list(datas) and all(ok), (what, "our decoder", rc, status)
    return stats


def hdr(st, kind, nbytes):
    return lit_header_bytes(st, kind)[nbytes]


# ---------------------------------------------------------------------------------------------------------------------
# the cases: name -> (inputs, [(edge, predicate over the list of per-frame statistics[, levels])])
def _raw_headers():
    ns = (31, 32, 4095, 4096)
    datas = [unique(n, 10 + n) * 2 for n in ns]  # n unmatchable literals, then one match of n at distance n
    checks = []
    for i, (n, h) in enumerate(zip(ns, (1, 2, 2, 3))):
        checks.append((f"Raw literals of {n} bytes with a {h}-byte header",
                       lambda S, i=i, n=n, h=h: hdr(S[i], "raw", h) == 1 and S[i]["regen_max_raw"] == n and S[i]["sequences"] == 1))
    return datas, checks


def _huf_headers():
    # literal-only frames (no 4-gram repeats: no sequences) of nlit skewed bytes; the last runs out of unseen 4-grams
    # and has a few short matches, but keeps more than 65536 literals
    ns = (255, 256, 1023, 1024, 16383, 16384, 70000)
    want = ((3, 1), (3, 4), (3, 4), (4, 4), (4, 4), (5, 4), (5, 4))  # (header bytes, streams)
    datas = [skewed(n, 20 + k) for k, n in enumerate(ns)]
    checks = []
    for i, (n, (h, s)) in enumerate(zip(ns, want)):
        sf = 0 if s == 1 else {3: 1, 4: 2, 5: 3}[h]
        checks.append((f"Huffman literals, nlit {n}: {s} stream(s), {h}-byte header",
                       lambda S, i=i, n=n, sf=sf: S[i]["lit_huf_sf" + str(sf)] == 1 and S[i]["regen_max_huf"] == S[i]["regen_min_huf"]
                       and (S[i]["regen_max_huf"] == n if n < 65536 else S[i]["regen_max_huf"] > 65536)))
    return datas, checks


def _huf_limit():
    # Geometric weights over 64 symbols (unmatchable) and Fibonacci weights over 26 (mostly matched away, the literals
    # left are still skewed): an unlimited tree would be far deeper than 11 levels; the first floor (total >> 11) is
    # enough for both.  The third input, 64 symbols of 300 and a Fibonacci chain 1, 1, 2 .. 377 below them with no
    # 4-gram twice (literals only: the histogram the encoder sees is the input's), needs the floor raised once.
    # Not covered: a second raise.  Every count is at least total / 2048 after the first floor, and the shapes that still
    # need two raises (a Fibonacci-like histogram over all symbols, e.g. L * (1, 1, 2 .. 610)) are dominated by a few
    # symbols whose 4-grams repeat: the match finder reduces them and no literal-only input of that shape was found.
    chain = exact_unique([300] * 64 + fib_weights(14), 1)
    raises = huf_floor_raises(chain)
    datas = [skewed(16_000, 31, nsym=64, q=0.85), unique(120_000, 32, 26, fib_weights(26)), chain]
    checks = [(f"Huffman code lengths limited to 11 bits (input {i})", lambda S, i=i: S[i]["huf_max_bits"] == 11) for i in range(3)]
    checks.append(("the Huffman floor raised once", lambda S: raises == 1 and S[2]["sequences"] == 0 and S[2]["lit_huf_sf3"] == 1))
    return datas, checks


def _weights():
    seen = set()
    direct = skewed(2000, 41, nsym=8, q=0.7)  # maxsym 7: seven direct weights are shorter than an FSE description
    fse_only = skewed(4000, 42, nsym=64, q=0.93, base=150)  # maxsym > 128: FSE-compressed weights
    sym255 = skewed(4000, 43, nsym=40, q=0.9, base=216)  # symbol 255 present
    all256 = bytes(unique(20_000, 44, 256, [40.0] + [1.0] * 255, seen=seen))  # every symbol, one frequent
    two = bytes(b & 1 for b in unique(30_000, 45, 256))  # symbols 0 and 1 only (nw = 1): a few hundred literals are left
    # maxsym 224 with 224 equally frequent symbols below it and the last at 1/8: every explicit weight is the same, which
    # neither description form can carry (direct: more than 128 weights; FSE: a single weight value) -> Raw literals,
    # although the codes would save 8 %
    eq = equal_weights()
    eq += eq[-60:]  # and one match, so that the block is not stored Raw as a whole
    datas = [direct, fse_only, sym255, all256, two, eq]
    checks = [
        ("direct weights (maxsym <= 128)", lambda S: S[0]["huf_wdirect"] >= 1 and S[0]["lit_huf_sf0"] + S[0]["lit_huf_sf1"] + S[0]["lit_huf_sf2"] >= 1),
        ("FSE-compressed weights (maxsym > 128)", lambda S: S[1]["huf_wfse"] >= 1 and S[1]["huf_wdirect"] == 0),
        ("Huffman literals with symbol 255", lambda S: S[2]["huf_max_sym"] == 255),
        ("Huffman literals over all 256 symbols", lambda S: S[3]["huf_max_nsym"] == 256),
        # (the greedy parse of level 1 matches all but a handful of these bytes)
        ("Huffman literals over two symbols (one explicit weight)", lambda S: S[4]["huf_wdirect"] >= 1 and S[4]["huf_min_nw"] == 1, (3, 9)),
        ("equal explicit weights above 128: Raw literals", lambda S: S[5]["huf_wfse"] + S[5]["huf_wdirect"] == 0 and S[5]["lit_raw"] >= 1
         and S[5]["regen_max_raw"] == len(eq) - 60),
    ]
    return datas, checks


def _nseq_headers():
    # The 3-byte form (0x7F00 = 32 512 sequences and more) takes a 128 KiB block of almost nothing but 4-byte matches
    # with no literals between them (the encoder stops at ZE_MAXSEQ - 32 = 32 736): grams_walk.  Only the greedy parse
    # of level 1 takes them one by one; the lazy parse of levels 3 and 9 prefers the longer match one byte later (the walk
    # is periodic) and writes a handful of long matches instead.
    datas = [with_sequences(127, 51), with_sequences(128, 53), with_sequences(5000, 53), grams_walk()]
    checks = [
        ("127 sequences: 1-byte Number_of_Sequences", lambda S: S[0]["sequences"] == 127 and S[0]["nseq_h1"] == 1),
        ("128 sequences: 2-byte Number_of_Sequences", lambda S: S[1]["sequences"] == 128 and S[1]["nseq_h2"] == 1),
        ("several thousand sequences: 2-byte Number_of_Sequences", lambda S: S[2]["sequences"] >= 4000 and S[2]["nseq_h2"] == 1),
        ("more than 0x7F00 sequences: 3-byte Number_of_Sequences", lambda S: S[3]["sequences"] > 0x7F00 and S[3]["nseq_h3"] == 1, (1,)),
    ]
    return datas, checks


P, R, F = "predefined", "rle", "fse"
COMBOS = [(P, P, P), (P, P, R), (P, R, R), (P, F, P), (P, F, R), (R, P, P), (R, P, R), (R, F, P), (R, F, R), (R, F, F), (F, F, R), (F, F, F)]


def _table_modes():
    # Fixed literal / match lengths give one LL / ML code (RLE_Mode); offsets kept within one code and never repeated
    # give one OF code; fewer than 64 (LL, ML) or 32 (OF) sequences leave a varied table Predefined, more make it FSE.
    # Covered: every (table x mode) pair, and the twelve (LL, OF, ML) combinations of COMBOS, which include one block
    # with a Predefined, an RLE and an FSE_Compressed table.  Not enumerated: the rest of the 27 triples.  Some the
    # heuristic hardly produces (LL or ML FSE needs 64 sequences or more, and then a varied OF table is Predefined only if
    # no offset code holds 1/16 of them); others it can (e.g. all three RLE) and are simply not among these inputs.
    # (the first literal run, 7 + 32 bytes, has the code of the others: 32..39)
    grid = [(k, lit, ml) for k in (20, 40, 300) for lit in ((32, 33), (12, 20)) for ml in ((5, 6), (5, 8))]
    datas = [with_sequences(k, 100 + i, lit, ml, new_offsets=True, first=7) for i, (k, lit, ml) in enumerate(grid)]
    datas.append(with_sequences(20, 102, (12, 20), (5, 6), new_offsets=True))  # offsets 29..44 within OF code 5

    def modes(s):
        return tuple(next(m for m in ("predefined", "rle", "fse") if s[f"{t}_{m}"]) for t in ("ll", "of", "ml"))

    checks = [
        ("one block with a Predefined, an RLE and an FSE_Compressed table", lambda S: any(len(set(modes(s))) == 3 for s in S)),
        *[(f"(LL, OF, ML) modes {c}", lambda S, c=c: any(modes(s) == c for s in S)) for c in COMBOS],
        *[(f"{t.upper()} table in {m} mode", lambda S, k=k, m=m: any(modes(s)[k] == m for s in S))
          for k, t in enumerate(("ll", "of", "ml")) for m in ("predefined", "rle", "fse")],
    ]
    return datas, checks


def _long_lengths():
    ll35 = run_then_match(70_000, 61)  # LL code 35
    ml52 = text(500, 62) + b"\x5a" * 70_000 + text(500, 63)  # one match of 69 999 at distance 1: ML code 52
    ll17 = run_then_match(BLOCK - 12, 64, back=100, ml=12)  # 131 060 literals and then a match at the block's very end
    checks = [
        ("literal run >= 65536 (LL code 35)", lambda S: S[0]["max_ll_code"] == 35 and S[0]["max_lit_run"] == 70_000),
        ("match >= 65539 (ML code 52)", lambda S: S[1]["max_ml_code"] == 52 and S[1]["max_match"] >= 65_539),
        ("literal run of 131060 in the 17-bit LL field", lambda S: S[2]["max_lit_run"] == BLOCK - 12 and S[2]["blocks"] == 1),
    ]
    return [ll35, ml52, ll17], checks


def _distance():
    # the run between the two copies of the phrase is one match at distance 1: the match finder's table is not
    # overwritten on the way (positions inside a match are never inserted)
    phrase = unique(64, 71)
    at = lambda d: phrase + b"\x00" * (d - 64) + phrase  # noqa: E731  (second copy exactly d bytes after the first)
    checks = [
        ("a repeat at distance 65535 is matched", lambda S: S[0]["max_offset"] == 65_535),
        ("a repeat at distance 65536 is not", lambda S: S[1]["max_offset"] < 65_535 and S[1]["regen_max_raw"] + S[1]["regen_max_huf"] >= 128),
        ("no offset beyond 65535 anywhere", lambda S: all(s["max_offset"] <= 65_535 for s in S)),
    ]
    return [at(65_535), at(65_536)], checks


def _blocks():
    t = text(3 * BLOCK, 81)
    sizes = (BLOCK - 1, BLOCK, BLOCK + 1, 2 * BLOCK + 1)
    datas = [t[:n] for n in sizes]
    datas.append(t[:BLOCK] + b"\x07" * BLOCK + t[:5000])  # a block of one byte inside a file
    datas.append(t[:BLOCK] + unique(BLOCK, 82) + t[:BLOCK])  # an incompressible block between compressed ones
    datas.append(t[:BLOCK] * 2 + t[:7000])  # the second block repeats the first: it must not reach back
    datas += [t[:n] for n in (255, 256, 65_791, 65_792)]
    checks = [(f"{n} bytes: {b} block(s)", lambda S, i=i, b=b: S[i]["blocks"] == b) for i, (n, b) in enumerate(zip(sizes, (1, 1, 2, 3)))]
    checks += [
        # the encoder writes Raw and Compressed blocks only: a block of one byte is one literal and one match
        ("a block of one byte: a literal and one match of 131071", lambda S: S[4]["max_match"] == BLOCK - 1 and S[4]["blocks_rle"] == 0),
        ("an incompressible block is stored Raw", lambda S: S[5]["blocks_raw"] == 1 and S[5]["blocks_compressed"] == 2),
        ("the repeat of a whole block is not matched across blocks", lambda S: S[6]["blocks"] == 3 and S[6]["xblock_matches"] == 0),
    ]
    for i, (n, f) in enumerate(zip((255, 256, 65_791, 65_792), (1, 2, 2, 4))):
        checks.append((f"{n} bytes: {f}-byte Frame_Content_Size", lambda S, i=i + 7, f=f: S[i]["fcs_size"] == f and S[i]["single_segment"] == 1))
    return datas, checks


def _chain_ranges():
    # Blocks of thousands of sequences whose codes are all common (no count-1 symbol for far more than the chain warm-up):
    # the FSE chain lanes start from a guessed state.  Valid frames here; bit-identity with the serial walk is checked by
    # the rare-path builds (tests/test_encoder_edges_emu.py).
    datas = [with_sequences(3000, 91), with_sequences(6000, 92, lit=(6, 8), ml=(4, 6))]
    return datas, [("thousands of sequences of a few codes", lambda S: all(s["sequences"] >= 2500 for s in S))]


CASES = {
    "raw_headers": _raw_headers,
    "huf_headers": _huf_headers,
    "huf_limit": _huf_limit,
    "weights": _weights,
    "nseq_headers": _nseq_headers,
    "table_modes": _table_modes,
    "long_lengths": _long_lengths,
    "distance": _distance,
    "blocks": _blocks,
    "chain_ranges": _chain_ranges,
}
_INPUTS = {}


def case_inputs(name):
    if name not in _INPUTS:
        _INPUTS[name] = CASES[name]()
    return _INPUTS[name]


def run_case(lib, name, levels=LEVELS, params=()):
    """all levels of one case; returns {level: (frames, stats)}"""
    datas, checks = case_inputs(name)
    out = {}
    for level in levels:
        frames = pack_frames(lib, datas, level, params)
        stats = check_frames(lib, datas, frames, (name, level))
        for edge, ok, *only in checks:  # (a third entry: the levels the edge is reachable at)
            if not only or level in only[0]:
                assert ok(stats), f"{name}, level {level}: the edge '{edge}' was not reached"
        # the encoder writes neither RLE literals nor RLE blocks (ze_literals_section, k_frame_assemble): a block's
        # literals hold every byte value of the block at least once, so they are one value only in a block of one value,
        # and that is one literal and one match
        assert all(st["lit_rle"] == 0 and st["blocks_rle"] == 0 for st in stats), (name, level, "RLE literals or blocks")
        out[level] = (frames, stats)
    return out


def run_cases(lib, names=None, levels=LEVELS):
    return {n: run_case(lib, n, levels) for n in (names or CASES)}

"""A Zstandard frame writer driven by an explicit description, and an executor that computes what the frame must
decode to from the same description (RFC 8878).  No libzstd: every mode, table and header form is whatever the
description says, so the decoder tests can reach frame shapes no encoder writes on purpose (tests/handmade_cases.py).

A frame description is a dict:

    blocks        list of block descriptions (below)
    single        Single_Segment_Flag (default True)
    window        Window_Descriptor byte when not single segment (default 0x58: 8 MiB)
    fcs           Frame_Content_Size field width in bytes: 0, 1, 2, 4, 8 or None for the smallest that fits
    fcs_value     the value written there (default: the regenerated size)
    did           (field width 0 / 1 / 2 / 4, value), default (0, 0)
    checksum      Content_Checksum_Flag (default False)

A block description is one of

    {"kind": "raw", "data": bytes}
    {"kind": "rle", "byte": int, "size": int}
    {"kind": "comp", "lit": literals, "seqs": [(literal_length, offset_value, match_length), ...],
     "ll" / "of" / "ml": table, "nseq_form": None | 1 | 2 | 3, "extra_bits": int}

literals = {"mode": "raw" | "rle" | "huf" | "treeless", "data": bytes, "streams": 1 | 4, "hdr": None | header bytes,
            "weights": None | list, "max_bits": 11, "wform": None | "direct" | "fse", "wlog": 6}
(Huffman weights are given, or derived from the byte counts of `data` under a code-length limit `max_bits`; the last
non-zero weight is the implicit one.  Treeless literals are coded with the tree of the last block that carried one, or
with `weights` when the description means to write an invalid frame.)

table = "pre" | ("rle", code) | ("fse", accuracy_log, normalized_counts) | "rep" | ("rep", table to code with)
(default "pre").  `extra_bits` > 0 leaves that many unread bits in the sequences bitstream, < 0 drops bits the
decoder needs.

`write(desc)` returns the frame; `execute(desc)` the bytes it regenerates, carrying the repeat-offset history across
blocks (RFC 8878 3.1.1.5) and raising ValueError for a description no valid frame can have.
"""
import heapq
import struct

LL_BASE = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40, 48, 64, 128, 256, 512, 1024,
           2048, 4096, 8192, 16384, 32768, 65536]
LL_BITS = [0] * 16 + [1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16]
ML_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 33,
           34, 35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051, 4099, 8195, 16387, 32771, 65539]
ML_BITS = [0] * 32 + [1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16]
LL_DEFAULT = (6, [4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1])
ML_DEFAULT = (6, [1, 4, 3, 2, 2, 2, 2, 2, 2] + [1] * 37 + [-1] * 7)
OF_DEFAULT = (5, [1, 1, 1, 1, 1, 1, 2, 2, 2] + [1] * 15 + [-1] * 5)
MAX_LOG = {"ll": 9, "of": 8, "ml": 9}
MAX_CODE = {"ll": 35, "of": 31, "ml": 52}
BLOCK_MAX = 128 * 1024


def seq(ll, offset, ml):
    """A sequence with a plain offset (never read as a repeat offset)."""
    return (ll, offset + 3, ml)


def highbit(v):
    return v.bit_length() - 1


def ll_code(v):
    return v if v < 16 else max(c for c in range(36) if LL_BASE[c] <= v)


def ml_code(v):
    return v - 3 if v < 35 else max(c for c in range(53) if ML_BASE[c] <= v)


# ---------------------------------------------------------------------------------------------------------------------
class BitWriter:
    """Little-endian bit writer: the first bit written is bit 0 of the first byte."""

    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.k = 0  # bits waiting in acc

    def put(self, value, nbits):
        assert 0 <= value < (1 << nbits) or (nbits == 0 and value == 0), (value, nbits)
        self.acc |= value << self.k
        self.k += nbits
        while self.k >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.k -= 8

    def forward_bytes(self):
        return bytes(self.out) + (bytes([self.acc]) if self.k else b"")

    def backward_bytes(self):
        """Closed with the 1-bit end marker: a decoder reading from the end sees the last field written first."""
        self.put(1, 1)
        return self.forward_bytes()


def backward_stream(fields):
    """fields in the order a decoder reads them -> the bitstream (written in reverse, then the marker)."""
    w = BitWriter()
    for value, nbits in reversed(fields):
        w.put(value, nbits)
    return w.backward_bytes()


# ---------------------------------------------------------------------------------------------------------------------
# FSE (RFC 8878 4.1.1)
class FseTable:
    """Decoding table of a distribution: per state (symbol, Number_of_Bits, Baseline); the encoder walks it backwards."""

    def __init__(self, log, norm):
        self.log, self.norm = log, list(norm)
        size = 1 << log
        assert sum(1 if c == -1 else c for c in norm) == size, ("counts do not fill the table", log, norm)
        sym = [None] * size
        high = size - 1
        for s, c in enumerate(norm):
            if c == -1:
                sym[high] = s
                high -= 1
        step, pos = (size >> 1) + (size >> 3) + 3, 0
        for s, c in enumerate(norm):
            for _ in range(max(c, 0)):
                sym[pos] = s
                pos = (pos + step) & (size - 1)
                while pos > high:
                    pos = (pos + step) & (size - 1)
        nxt = [1 if c == -1 else c for c in norm]
        self.states = []
        self.by_sym = {}
        for i in range(size):
            s = sym[i]
            x = nxt[s]
            nxt[s] += 1
            nb = log - highbit(x)
            base = (x << nb) - size
            self.states.append((s, nb, base))
            self.by_sym.setdefault(s, []).append(i)

    def prev_state(self, s, following):
        """The state that decodes symbol s and whose update lands on state `following` -> (state, bits read)."""
        for i in self.by_sym[s]:
            _, nb, base = self.states[i]
            if base <= following < base + (1 << nb):
                return i, following - base
        raise AssertionError("FSE state intervals must cover the table")

    def encode_chain(self, syms):
        """Decoder states for syms (the last state is the first one with the last symbol) and the update bits
        [(value, nbits)] read after each symbol but the last."""
        for s in syms:
            if s not in self.by_sym:
                raise ValueError(f"symbol {s} has probability 0 in this table")
        states = [self.by_sym[syms[-1]][0]]
        upd = []
        for s in reversed(syms[:-1]):
            i, bits = self.prev_state(s, states[-1])
            upd.append((bits, self.states[i][1]))
            states.append(i)
        states.reverse()
        upd.reverse()
        return states, upd


class RleTable:
    log = 0

    def __init__(self, code):
        self.code = code
        self.by_sym = {code: [0]}

    def encode_chain(self, syms):
        if any(s != self.code for s in syms):
            raise ValueError("an RLE table codes one symbol")
        return [0] * len(syms), [(0, 0)] * (len(syms) - 1)


def ncount_bits(w, log, norm):
    """NCount (RFC 8878 4.1.1): accuracy log - 5, then the counts with the repeat-zero flags, written to w."""
    norm = list(norm)
    while norm and norm[-1] == 0:
        norm.pop()
    w.put(log - 5, 4)
    remaining = 1 << log
    s = 0
    while remaining > 0:
        assert s < len(norm), "counts end before the table is full"
        p = norm[s]
        bits = highbit(remaining + 1) + 1
        thr = (1 << bits) - 1 - (remaining + 1)
        val = p + 1
        half = 1 << (bits - 1)
        if val < thr:
            w.put(val, bits - 1)
        elif val < half:
            w.put(val, bits)
        else:
            w.put((val - half + thr) | half, bits)
        remaining -= 1 if p < 0 else p
        s += 1
        if p == 0:
            z = 0
            while s + z < len(norm) and norm[s + z] == 0:
                z += 1
            s += z
            while z >= 3:
                w.put(3, 2)
                z -= 3
            w.put(z, 2)
    assert remaining == 0 and s == len(norm), ("counts overfill the table", log, norm)


def ncount_bytes(log, norm):
    w = BitWriter()
    ncount_bits(w, log, norm)
    return w.forward_bytes()


def normalize(counts, log):
    """counts (list, 0 = absent) -> normalized counts summing to 2^log, every present symbol >= 1."""
    size = 1 << log
    total = sum(counts)
    norm = [max(1, c * size // total) if c else 0 for c in counts]
    while sum(norm) > size:
        i = max(range(len(norm)), key=lambda k: norm[k])
        norm[i] -= 1
    while sum(norm) < size:
        i = max(range(len(norm)), key=lambda k: counts[k])
        norm[i] += 1
    return norm


# ---------------------------------------------------------------------------------------------------------------------
# Huffman (RFC 8878 4.2)
def huffman_lengths(counts, limit):
    """Code lengths (0 = absent) of a Huffman code for counts, no length above `limit` (counts are flattened until the
    tree fits).  At least two symbols are present."""
    counts = list(counts)
    assert sum(1 for c in counts if c) <= 1 << limit, "more symbols than codes of that length"
    while True:
        heap = [(c, i, (i,)) for i, c in enumerate(counts) if c]
        assert len(heap) >= 2, "a Huffman code needs two symbols"
        heapq.heapify(heap)
        depth = [0] * len(counts)
        tie = len(counts)
        while len(heap) > 1:
            c1, _, a = heapq.heappop(heap)
            c2, _, b = heapq.heappop(heap)
            for s in a + b:
                depth[s] += 1
            heapq.heappush(heap, (c1 + c2, tie, a + b))
            tie += 1
        if max(depth) <= limit:
            return depth
        counts = [(c + 1) // 2 if c else 0 for c in counts]


def weights_from_data(data, limit=11, extra=()):
    counts = [0] * 256
    for b in data:
        counts[b] += 1
    for b in extra:
        counts[b] += 1
    if sum(1 for c in counts if c) < 2:
        counts[(max(data) + 1) % 256 if data else 1] += 1
    lengths = huffman_lengths(counts, limit)
    max_len = max(lengths)
    w = [max_len + 1 - n if n else 0 for n in lengths]
    while w[-1] == 0:
        w.pop()
    return w


class HufCode:
    """Canonical code of a weight list (RFC 8878 4.2.1): symbol -> (code, length)."""

    def __init__(self, weights):
        self.weights = list(weights)
        total = sum(1 << (x - 1) for x in weights if x)
        self.max_bits = highbit(total)
        assert total == 1 << self.max_bits, "weights must describe a complete code"
        rank_start = {}
        pos = 0
        for wv in range(1, 13):
            rank_start[wv] = pos
            pos += sum(1 for x in weights if x == wv) << (wv - 1)
        self.code = {}
        for s, x in enumerate(weights):
            if x:
                nb = self.max_bits + 1 - x
                self.code[s] = (rank_start[x] >> (x - 1), nb)
                rank_start[x] += 1 << (x - 1)

    def stream(self, data):
        try:
            return backward_stream([self.code[b] for b in data])
        except KeyError as e:
            raise ValueError(f"byte {e} has no Huffman code") from None


def weights_direct(weights):
    ex = list(weights[:-1])
    assert 1 <= len(ex) <= 128
    if len(ex) & 1:
        ex.append(0)
    return bytes([127 + len(weights) - 1]) + bytes((ex[i] << 4) | ex[i + 1] for i in range(0, len(ex), 2))


def weights_fse(weights, log=6):
    """The explicit weights coded with FSE: two interleaved states, the stream ending where the update after the
    next-to-last weight runs past its start (RFC 8878 4.2.1.2)."""
    ex = list(weights[:-1])
    assert len(ex) >= 2
    counts = [0] * 12
    for x in ex:
        counts[x] += 1
    if sum(1 for c in counts if c) < 2:  # one value: a second one in the table gives the states a bit to read
        counts[1 if ex[0] != 1 else 2] += 1
    t = FseTable(log, normalize(counts, log))
    m = len(ex)
    a, b = ex[0::2], ex[1::2]
    # the chain holding weight m-2 ends with an update that must read at least one bit (that read runs dry)
    pen = a if (m - 2) % 2 == 0 else b
    last_state = next((i for i in t.by_sym[pen[-1]] if t.states[i][1] > 0), None)
    assert last_state is not None
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
    for j in range(m - 2):  # the update after weight j (chain j % 2, its (j // 2)-th)
        fields.append(chains[j % 2][1][j // 2])
    body = ncount_bytes(log, t.norm) + backward_stream(fields)
    assert len(body) < 128, "FSE-coded weights take 127 bytes at most"
    return bytes([len(body)]) + body


# ---------------------------------------------------------------------------------------------------------------------
def lit_header(ltype, regen, comp, streams, hdr):
    if ltype < 2:
        fits = [h for h, lim in ((1, 31), (2, 4095), (3, (1 << 20) - 1)) if regen <= lim]
        h = hdr or fits[0]
        if h == 1:
            return bytes([ltype | (regen << 3) & 0xFF])
        if h == 2:
            return struct.pack("<H", ltype | 1 << 2 | regen << 4)
        return struct.pack("<I", ltype | 3 << 2 | regen << 4)[:3]
    if hdr is None:
        hdr = 3 if max(regen, comp) < 1024 else 4 if max(regen, comp) < 16384 else 5
    if hdr == 3:
        sf = 0 if streams == 1 else 1
        return struct.pack("<I", ltype | sf << 2 | regen << 4 | comp << 14)[:3]
    assert streams == 4, "the 4- and 5-byte headers are for 4 streams"
    if hdr == 4:
        return struct.pack("<I", ltype | 2 << 2 | regen << 4 | comp << 18)
    return struct.pack("<Q", ltype | 3 << 2 | regen << 4 | comp << 22)[:5]


def nseq_bytes(n, form):
    form = form or (1 if n < 128 else 2 if n < 0x7F00 else 3)
    if form == 1:
        assert n < 128
        return bytes([n])
    if form == 2:
        assert n < 0x7F00
        return bytes([(n >> 8) + 128, n & 255])
    assert n >= 0x7F00
    return bytes([255]) + struct.pack("<H", n - 0x7F00)


def _table(kind, spec, prev):
    """-> (mode, description bytes, table)"""
    if spec is None or spec == "pre":
        log, norm = {"ll": LL_DEFAULT, "of": OF_DEFAULT, "ml": ML_DEFAULT}[kind]
        return 0, b"", FseTable(log, norm)
    if spec == "rep" or spec[0] == "rep":
        t = prev if spec == "rep" else _table(kind, spec[1], None)[2]
        if t is None:
            raise ValueError(f"Repeat_Mode for {kind} with no earlier table (give one to code with)")
        return 3, b"", t
    if spec[0] == "rle":
        return 1, bytes([spec[1]]), RleTable(spec[1])
    _, log, norm = spec
    return 2, ncount_bytes(log, norm), FseTable(log, norm)


def _literals(lit, state):
    mode, data = lit["mode"], bytes(lit["data"])
    if mode == "raw":
        return lit_header(0, lit.get("size", len(data)), 0, 1, lit.get("hdr")) + data  # ("size": a false header)
    if mode == "rle":
        assert data and len(set(data)) == 1, "RLE literals repeat one byte"
        return lit_header(1, len(data), 0, 1, lit.get("hdr")) + data[:1]
    tree = b""
    if mode == "huf":
        weights = lit.get("weights") or weights_from_data(data, lit.get("max_bits", 11))
        wform = lit.get("wform") or ("direct" if len(weights) - 1 <= 128 else "fse")
        tree = weights_direct(weights) if wform == "direct" else weights_fse(weights, lit.get("wlog", 6))
        code = HufCode(weights)
        state["huf"] = code
    else:
        code = HufCode(lit["weights"]) if lit.get("weights") else state.get("huf")
        if code is None:
            raise ValueError("Treeless literals with no earlier tree (give weights to code with)")
    streams = lit.get("streams", 1)
    if streams == 1:
        body = tree + code.stream(data)
    else:
        seg = (len(data) + 3) // 4
        parts = [code.stream(data[i * seg : (i + 1) * seg] if i < 3 else data[3 * seg :]) for i in range(4)]
        body = tree + struct.pack("<HHH", *(len(p) for p in parts[:3])) + b"".join(parts)
    return lit_header(2 if mode == "huf" else 3, len(data), len(body), streams, lit.get("hdr")) + body


def _compressed_block(b, state):
    out = bytearray(_literals(b["lit"], state))
    seqs = b.get("seqs", [])
    out += nseq_bytes(len(seqs), b.get("nseq_form"))
    if not seqs:
        return bytes(out)
    modes, tables = 0, {}
    for kind, shift in (("ll", 6), ("of", 4), ("ml", 2)):
        mode, desc, t = _table(kind, b.get(kind), state.get(kind))
        modes |= mode << shift
        tables[kind] = t
        state[kind] = t
    out.append(modes)
    for kind in ("ll", "of", "ml"):
        spec = b.get(kind)
        if spec and spec not in ("pre", "rep") and spec[0] in ("rle", "fse"):
            out += _table(kind, spec, None)[1]
    lc = [ll_code(s[0]) for s in seqs]
    oc = [highbit(s[1]) for s in seqs]
    mc = [ml_code(s[2]) for s in seqs]
    ch = {k: tables[k].encode_chain(c) for k, c in (("ll", lc), ("of", oc), ("ml", mc))}
    fields = [(ch["ll"][0][0], tables["ll"].log), (ch["of"][0][0], tables["of"].log), (ch["ml"][0][0], tables["ml"].log)]
    for i, (ll, ov, ml) in enumerate(seqs):
        fields.append((ov - (1 << oc[i]), oc[i]))
        fields.append((ml - ML_BASE[mc[i]], ML_BITS[mc[i]]))
        fields.append((ll - LL_BASE[lc[i]], LL_BITS[lc[i]]))
        if i + 1 < len(seqs):
            fields += [ch["ll"][1][i], ch["ml"][1][i], ch["of"][1][i]]
    extra = b.get("extra_bits", 0)
    if extra > 0:
        fields.append((0, extra))
    elif extra < 0:
        drop = -extra
        while drop:  # the last fields read lose their bits
            v, n = fields.pop()
            if n > drop:
                fields.append((v >> drop, n - drop))
                drop = 0
            else:
                drop -= n
    out += backward_stream(fields)
    return bytes(out)


def nominal_size(desc):
    """Bytes the blocks claim to regenerate (exact for valid descriptions)."""
    n = 0
    for b in desc["blocks"]:
        if b["kind"] == "raw":
            n += len(b["data"])
        elif b["kind"] == "rle":
            n += b["size"]
        else:
            n += len(b["lit"]["data"]) + sum(s[2] for s in b.get("seqs", []))
    return n


def write(desc):
    import xxhash

    single = desc.get("single", True)
    size = nominal_size(desc)
    fcs_value = desc.get("fcs_value", size)
    width = desc.get("fcs")
    if width is None:
        width = (1 if single else 0) if fcs_value < 256 else 2 if fcs_value < 65536 + 256 else 4 if fcs_value < 1 << 32 else 8
    did_w, did = desc.get("did", (0, 0))
    flag = {0: 0, 1: 0, 2: 1, 4: 2, 8: 3}[width]
    assert (width == 0 and not single) or (width == 1 and single) or width >= 2
    out = bytearray(struct.pack("<I", 0xFD2FB528))
    out.append(flag << 6 | single << 5 | desc.get("checksum", False) << 2 | {0: 0, 1: 1, 2: 2, 4: 3}[did_w])
    if not single:
        out.append(desc.get("window", 0x58))
    out += did.to_bytes(did_w, "little")
    if width:
        out += (fcs_value - (256 if width == 2 else 0)).to_bytes(width, "little")
    state = {}
    blocks = desc["blocks"]
    for i, b in enumerate(blocks):
        last = i + 1 == len(blocks)
        if b["kind"] == "raw":
            body, typ, bsize = bytes(b["data"]), 0, len(b["data"])
        elif b["kind"] == "rle":
            body, typ, bsize = bytes([b["byte"]]), 1, b["size"]
        else:
            body = _compressed_block(b, state)
            typ, bsize = 2, len(body)
        out += struct.pack("<I", last | typ << 1 | bsize << 3)[:3] + body
    if desc.get("checksum"):
        content = execute(desc) if desc.get("valid", True) else bytes(size)
        out += struct.pack("<I", xxhash.xxh64(content, seed=0).intdigest() & 0xFFFFFFFF)
    return bytes(out)


def resolve(rep, ll, ov):
    """Offset_Value -> (offset, new repeat history) (RFC 8878 3.1.1.5)."""
    if ov > 3:
        return ov - 3, [ov - 3, rep[0], rep[1]]
    idx = ov - 1 + (ll == 0)
    if idx == 0:
        return rep[0], rep
    off = rep[0] - 1 if idx == 3 else rep[idx]
    if off == 0:
        raise ValueError("repeat offset rep0 - 1 of 1")
    return off, [off, rep[0], rep[2] if idx == 1 else rep[1]]


def execute(desc):
    """The bytes the frame regenerates (RFC 8878 3.1.1.4-3.1.1.5), from the description alone."""
    out = bytearray()
    rep = [1, 4, 8]
    for b in desc["blocks"]:
        start = len(out)
        if b["kind"] == "raw":
            out += b["data"]
        elif b["kind"] == "rle":
            out += bytes([b["byte"]]) * b["size"]
        else:
            lits = bytes(b["lit"]["data"])
            pos = 0
            for ll, ov, ml in b.get("seqs", []):
                if ml < 3 or ov < 1:
                    raise ValueError("match length < 3 or offset value 0")
                off, rep = resolve(rep, ll, ov)
                if pos + ll > len(lits):
                    raise ValueError("sequences consume more literals than the block has")
                out += lits[pos : pos + ll]
                pos += ll
                if off > len(out):
                    raise ValueError("a match reaches before the frame's start")
                for _ in range(ml):
                    out.append(out[-off])
            out += lits[pos:]
        if len(out) - start > BLOCK_MAX:
            raise ValueError("a block regenerates more than 128 KiB")
    return bytes(out)

"""Negative compression levels: libzstd's fast strategy with an acceleration of -level, Raw literals in every block, and
from -2 down the strided parse of the match finder (zstd_encode.cu: ze_resolve_params, ze_fast_block).

Shared by the CPU suite (tests/test_fast_levels_emu.py) and the GPU suite (tests/test_fast_levels_gpu.py).  Every check
is a function of the library under test and raises AssertionError naming what went wrong."""
import ctypes as C

import numpy as np

from oracle import ref_path
from tests import encoder_edge_cases as E
from tests.golden.recipes import text
from tests.helpers import layout, pack_batch

LEVELS = (-1, -2, -3, -5, -10, -50, -131072)
BLOCK = 131072


# ---------------------------------------------------------------------------------------------------------------------
# inputs
def c2_batch(lib, total_bytes, seed=21):
    from zarc_b200 import corpus

    c = corpus.c2_source_tree(total_bytes=total_bytes, seed=seed)
    blob = corpus.materialise_host(lib, c)
    return [bytes(blob[int(o) : int(o) + int(n)]) for o, n in zip(c.off, c.len)]


def log_lines(n, seed):
    """a multi-block server log: timestamps, a few levels and paths, numbers"""
    rng = np.random.default_rng(seed)
    words = [b"GET", b"POST", b"/api/v1/items", b"/static/app.js", b"/login", b"INFO", b"WARN", b"ERROR", b"user", b"session"]
    out = bytearray()
    t = 1_700_000_000
    while len(out) < n:
        t += int(rng.integers(0, 5))
        parts = [str(t).encode(), words[int(rng.integers(5, 8))], *(words[int(k)] for k in rng.integers(0, 10, 3)),
                 str(int(rng.integers(0, 100000))).encode(), b"%d ms" % int(rng.integers(1, 900))]
        out += b" ".join(parts) + b"\n"
    return bytes(out[:n])


def edge_inputs():
    """the small and boundary-sized files, and inputs whose literals sections need Raw headers of 1, 2 and 3 bytes"""
    raw_hdr = [E.unique(k, 10 + k) * 2 for k in (31, 32, 4095, 4096)]  # k unmatchable literals, then one match of k
    sized = [b"", b"a", text(15, 1), text(16, 2), text(BLOCK, 3), text(BLOCK + 1, 4)]
    return sized + raw_hdr + [log_lines(1 << 20, 5), np.random.default_rng(6).bytes(300_000)]


# ---------------------------------------------------------------------------------------------------------------------
# the frames
def pack(lib, datas, level, params=(), init=0):
    """one frame per input through zg_pack_batch; `init`: the level given to zg_cctx_init (the parameter is then not set
    when `level` is None)"""
    cctx = lib.zg_cctx_create()
    try:
        lib.check(lib.zg_cctx_init(cctx, init))
        lib.check(lib.zg_cctx_set_parameter(cctx, 201, 1))
        if level is not None:
            lib.check(lib.zg_cctx_set_parameter(cctx, 100, level))
        for p, v in params:
            lib.check(lib.zg_cctx_set_parameter(cctx, p, v))
        lib.check(lib.zg_cctx_reset_archive(cctx, 12))
        r = pack_batch(lib, cctx, datas)
    finally:
        lib.zg_cctx_free(cctx)
    assert r["rc"] == 0, r["rc"]
    return [bytes(r["frames"][o - 12 : o - 12 + ln]) for o, ln in zip(r["off"], r["len"])]


def blocks(frame):
    """[(Block_Type, body)] of a frame, in order"""
    fhd = frame[4]
    did = {0: 0, 1: 1, 2: 2, 3: 4}[fhd & 3]
    fcs = {0: 1 if fhd & 0x20 else 0, 1: 2, 2: 4, 3: 8}[fhd >> 6]
    p = 5 + (0 if fhd & 0x20 else 1) + did + fcs
    out = []
    while True:
        h = int.from_bytes(frame[p : p + 3], "little")
        last, btype, size = h & 1, (h >> 1) & 3, h >> 3
        body = frame[p + 3 : p + 3 + (1 if btype == 1 else size)]
        out.append((btype, body))
        p += 3 + len(body)
        if last:
            return out


def sequences_section(body):
    """the sequences section of a Compressed block's body: what follows its literals section"""
    ltype, sf = body[0] & 3, (body[0] >> 2) & 3
    if ltype in (0, 1):
        hl = {0: 1, 2: 1, 1: 2, 3: 3}[sf]
        regen = int.from_bytes(body[:hl], "little") >> (3 if hl == 1 else 4)
        return body[hl + (regen if ltype == 0 else 1) :]
    hl, cbits = {0: (3, 10), 1: (3, 10), 2: (4, 14), 3: (5, 18)}[sf]
    comp = (int.from_bytes(body[:hl], "little") >> (4 + cbits)) & ((1 << cbits) - 1)
    return body[hl + comp :]


def nseq(body):
    s = sequences_section(body)
    return s[0] if s[0] < 128 else ((s[0] - 128) << 8) + s[1] if s[0] < 255 else s[1] + (s[2] << 8) + 0x7F00


def check_frames(lib, datas, frames, what):
    """every decoder restores every frame (checksums verified), Frame_Content_Size is the input's size, no literals
    section is Huffman, Treeless or RLE; returns the C oracle's statistics"""
    stats = E.check_frames(lib, datas, frames, what)
    for i, (d, fr) in enumerate(zip(datas, frames)):
        assert ref_path._zstd.ZSTD_getFrameContentSize(fr, len(fr)) == len(d), (what, i, "Frame_Content_Size")
        st = stats[i]
        assert st["has_checksum"] == 1, (what, i)
        assert st["lit_huf1"] + st["lit_huf4"] + st["lit_treeless"] + st["lit_rle"] == 0, (what, i, "compressed literals")
    return stats


# ---------------------------------------------------------------------------------------------------------------------
# the checks
def run_levels(lib, datas, c2_count):
    """Round trips and every property of the parses on `datas`, whose first `c2_count` inputs are the C2-shaped batch.
    Returns {level: total frame bytes} of ours and libzstd's."""
    ours, ref = {}, {}
    frames1 = pack(lib, datas, 1)
    for lv in LEVELS:
        frames = pack(lib, datas, lv)
        stats = check_frames(lib, datas, frames, lv)
        ours[lv] = sum(map(len, frames))
        if lv in (-1, -3, -5, -10):
            ref[lv] = sum(len(ref_path.ref_compress(d, level=lv)) for d in datas)
        if lv == -1:
            # the parse of level 1 with Raw literals: equal sequences sections wherever both levels compressed a block
            same = 0
            for i, (a, b) in enumerate(zip(frames, frames1)):
                for j, ((ta, ba), (tb, bb)) in enumerate(zip(blocks(a), blocks(b))):
                    if ta == 2 and tb == 2:
                        assert sequences_section(ba) == sequences_section(bb), (i, j, "sequences at -1 and 1 differ")
                        same += 1
            assert same >= c2_count // 2, same
            # Raw literals headers of 1, 2 and 3 bytes, each reached
            seen = {h: sum(E.lit_header_bytes(st, "raw")[h] for st in stats) for h in (1, 2, 3)}
            assert all(seen.values()), seen
        else:
            for i, st in enumerate(stats):
                if st["sequences"]:
                    assert st["min_match"] >= 4 and st["max_offset"] <= 65535, (lv, i, st["min_match"], st["max_offset"])
        if lv == -131072:
            for i, fr in enumerate(frames):
                for t, body in blocks(fr):
                    assert t == 0 or (t == 2 and nseq(body) <= 1), (i, t)
            assert all(st["blocks_compressed"] == 0 for st in stats[:c2_count]), "a C2 block is not Raw at -131072"
    # the knob: lower levels never give smaller archives
    sizes = [ours[lv] for lv in (-1, -2, -3, -5, -10, -50)]
    assert sizes == sorted(sizes), sizes
    # against libzstd at the same level: within 10 % at -1, -3 and -5.  -10 misses that bound (1.14 on these inputs:
    # libzstd also probes the last offset at every step and adds positions around each match to its table, this parse
    # does neither); its factor is returned for the caller to report, not held to a bound of its own
    factors = {lv: ours[lv] / ref[lv] for lv in ref}
    assert all(factors[lv] <= 1.10 for lv in (-1, -3, -5)), factors
    return ours, ref, factors


def check_combinations(lib, datas):
    """strategy >= 2 or searchLog turn fast mode off (the level then acts as level 1); zg_cctx_init(-5) and
    set_parameter(level, -5) are one setting, and the setter returns 0 as libzstd's does"""
    for p, v in ((107, 2), (104, 2)):
        assert pack(lib, datas, -5, [(p, v)]) == pack(lib, datas, 1, [(p, v)]), (p, v)
    assert pack(lib, datas, None, init=-5) == pack(lib, datas, -5)
    cctx = lib.zg_cctx_create()
    try:
        assert lib.zg_cctx_set_parameter(cctx, 100, -5) == 0
        assert lib.zg_cctx_set_parameter(cctx, 100, -131072) == 0
        assert lib.zg_is_error(lib.zg_cctx_set_parameter(cctx, 100, -131073))
        assert lib.zg_is_error(lib.zg_cctx_set_parameter(cctx, 106, 5))  # targetLength stays refused
    finally:
        lib.zg_cctx_free(cctx)


def check_fast_parameters(lib, datas):
    """windowLog, minMatch and hashLog keep their meaning in the strided parse: at -5 with windowLog 10 and minMatch 6
    no offset exceeds 1024 and no match is shorter than 6, and a table of 2^8 positions finds less than the default"""
    frames = pack(lib, datas, -5, [(101, 10), (105, 6)])
    stats = check_frames(lib, datas, frames, "-5, windowLog 10, minMatch 6")
    assert sum(st["sequences"] for st in stats) > 0
    for i, st in enumerate(stats):
        if st["sequences"]:
            assert st["max_offset"] <= 1024 and st["min_match"] >= 6, (i, st["max_offset"], st["min_match"])
    default = pack(lib, datas, -5)
    assert sum(map(len, frames)) > sum(map(len, default))
    small = pack(lib, datas, -5, [(102, 8)])
    check_frames(lib, datas, small, "-5, hashLog 8")
    assert sum(map(len, small)) > sum(map(len, default))


def pack_dev(lib, datas, level, to_dev, to_host):
    """zg_pack_batch_dev: inputs and outputs in device memory (`to_dev`: numpy -> (keep-alive object, address);
    `to_host`: keep-alive object -> numpy)"""
    blob, off, lens = layout(datas)
    n = len(datas)
    cap = int(lens.sum()) + 1024 + 64 * n
    bufs = {k: to_dev(a) for k, a in (("blob", blob), ("off", off), ("len", lens), ("dig", np.zeros(32 * n, np.uint8)),
                                       ("first", np.zeros(n, np.uint8)), ("foff", np.zeros(n, np.uint64)), ("flen", np.zeros(n, np.uint64)),
                                       ("frames", np.zeros(cap, np.uint8)))}
    nbytes = np.zeros(1, dtype=np.uint64)
    cctx = lib.zg_cctx_create()
    try:
        lib.check(lib.zg_cctx_init(cctx, 0))
        lib.check(lib.zg_cctx_set_parameter(cctx, 201, 1))
        lib.check(lib.zg_cctx_set_parameter(cctx, 100, level))
        lib.check(lib.zg_cctx_reset_archive(cctx, 12))
        a = {k: v[1] for k, v in bufs.items()}
        lib.check(lib.zg_pack_batch_dev(cctx, a["blob"], a["off"], a["len"], n, a["dig"], a["first"], a["foff"], a["flen"], a["frames"], cap,
                                        nbytes.ctypes.data))
    finally:
        lib.zg_cctx_free(cctx)
    arch = to_host(bufs["frames"][0])[: int(nbytes[0])].tobytes()
    foff, flen = (np.ascontiguousarray(to_host(bufs[k][0])).view(np.uint64).astype(np.int64) for k in ("foff", "flen"))
    return [arch[o - 12 : o - 12 + ln] for o, ln in zip(foff, flen)]


def check_paths(lib, datas, to_dev=None, to_host=None, level=-5):
    """the same frames from the sliced host path, the device path, a small encoder chunk, and with every file repeated
    within a call and across calls (dedup)"""
    want = pack(lib, datas, level)
    if to_dev is not None:
        assert pack_dev(lib, datas, level, to_dev, to_host) == want, "zg_pack_batch_dev"
    try:
        for slice_bytes, chunk_bytes in ((70_000, 0), (0, 65536), (33_000, 4096)):
            lib.dll.zg_internal_set_slice_bytes(C.c_uint64(slice_bytes))
            lib.dll.zg_internal_set_encode_chunk_bytes(C.c_uint64(chunk_bytes))
            assert pack(lib, datas, level) == want, (slice_bytes, chunk_bytes)
    finally:
        lib.dll.zg_internal_set_slice_bytes(C.c_uint64(0))
        lib.dll.zg_internal_set_encode_chunk_bytes(C.c_uint64(0))
    # dedup: repeats within a call point at the first frame, and a second call finds them all
    cctx = lib.zg_cctx_create()
    try:
        lib.check(lib.zg_cctx_init(cctx, level))
        lib.check(lib.zg_cctx_set_parameter(cctx, 201, 1))
        lib.check(lib.zg_cctx_reset_archive(cctx, 12))
        r = pack_batch(lib, cctx, datas + datas[::-1])
        assert r["rc"] == 0
        uniq = {}
        for d, o, ln, f in zip(datas + datas[::-1], r["off"], r["len"], r["first"]):
            fr = bytes(r["frames"][o - 12 : o - 12 + ln])
            assert uniq.setdefault(d, fr) == fr
        assert [uniq[d] for d in datas] == want
        r2 = pack_batch(lib, cctx, datas)
        assert r2["rc"] == 0 and not any(r2["first"]) and r2["frames"] == b""
    finally:
        lib.zg_cctx_free(cctx)

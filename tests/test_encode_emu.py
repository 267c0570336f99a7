"""K2/K3 encoder + pack bookkeeping on the SIMT emulator.  GPU-made frames must be valid Zstandard
that the reference decoder (libzstd 1.5.5, one-shot AND the reference's streaming call sequence)
restores byte-identically; dedup decisions, offsets and digests must equal the reference path's."""
import numpy as np
import pytest

from oracle import ref_path
from tests.golden.recipes import RECIPES, make_input, text, rand
from tests.helpers import compress2, pack_batch, unpack_batch


def _check_frame(lib, data, frame):
    assert ref_path.ref_decompress(frame, len(data)) == data  # libzstd one-shot
    assert ref_path.ref_decompress_stream(b"\x00" * 5 + frame + b"tail", 5) == data  # zstd_iterator.rs call sequence
    got, err, consumed, _ = ref_path.c_zstd_decompress_frame(frame, len(data))  # C restatement
    assert err == 0 and got == data and consumed == len(frame)
    assert ref_path.find_frame_compressed_size(frame) == len(frame)


@pytest.mark.parametrize("name", list(RECIPES))
def test_compress2_recipes(emu, name):
    data = make_input(name)
    for level in (1, 3):
        frame = compress2(emu, data, level=level)
        _check_frame(emu, data, frame)
        assert len(frame) <= emu.zg_compress_bound(len(data))


def test_compress2_known_answer_shapes(emu):
    # empty / tiny inputs are single Raw blocks exactly like libzstd's (SURVEY.md App. E)
    assert compress2(emu, b"").hex() == "28b52ffd2400010000" + "99e9d851"
    assert compress2(emu, b"a").hex() == "28b52ffd2401090000" + "61" + "5b6e8ca9"
    assert compress2(emu, b"hello world\n").hex() == "28b52ffd240c610000" + b"hello world\n".hex() + "8c6d7d20"
    assert compress2(emu, b"a", checksum=False).hex() == "28b52ffd2001090000" + "61"


def test_compress2_flags_and_errors(emu):
    import ctypes as C

    data = text(30000, 5)
    f = compress2(emu, data, checksum=False, content_size=False)
    _check_frame(emu, data, f)
    c = emu.zg_cctx_create()
    assert emu.zg_cctx_set_parameter(c, 201, 1) == 1  # returns the value set, like libzstd
    assert emu.zg_get_error_code(emu.zg_cctx_set_parameter(c, 100, 99)) == 42
    assert emu.zg_get_error_code(emu.zg_cctx_set_parameter(c, 9999, 1)) == 40
    rnd = rand(5000, 1)
    small = C.create_string_buffer(100)
    assert emu.zg_get_error_code(emu.zg_compress2(c, small, 100, rnd, len(rnd))) == 70  # never overruns
    assert small.raw[99:] == b"\x00"
    emu.zg_cctx_free(c)


def few_sequence_inputs():
    """Blocks with 1, 2, 3 ... a few dozen sequences (the FSE state chains are cut into ten ranges per chain: every
    count around that has to come out right), blocks made of one repeated phrase (RLE sequence tables), and blocks whose
    sequence codes are all distinct (count-1 symbols everywhere)."""
    rng = np.random.default_rng(2024)
    phrase = rand(37, 3)
    out = []
    for k in range(1, 48):  # k phrases re-used once each, separated by fresh bytes: about k sequences
        parts = []
        for j in range(k):
            parts.append(rand(int(rng.integers(9, 30)), 100 * k + j))
            parts.append(phrase[: int(rng.integers(8, 37))])
        out.append(phrase + b"".join(parts))
    out.append((phrase + rand(5, 9)) * 300)                      # identical sequences: RLE tables
    out.append(b"".join(rand(6 + j % 40, j) + phrase[: 5 + j % 30] for j in range(400)))  # varied lengths and offsets
    out.append(text(3000, 77) + bytes(4000) + text(3000, 77))    # long match, long zero run
    return out


@pytest.mark.parametrize("level", [1, 3])
def test_few_sequences_and_chain_ranges(emu, level):
    datas = few_sequence_inputs()
    cctx = emu.zg_cctx_create()
    emu.check(emu.zg_cctx_init(cctx, level))
    emu.check(emu.zg_cctx_set_parameter(cctx, 201, 1))
    emu.check(emu.zg_cctx_reset_archive(cctx, 12))
    r = pack_batch(emu, cctx, datas)
    emu.zg_cctx_free(cctx)
    assert r["rc"] == 0
    for d, o, l in zip(datas, r["off"], r["len"]):
        _check_frame(emu, d, bytes(r["frames"][o - 12 : o - 12 + l]))


def test_ratio_vs_reference_small_corpus(emu):
    from zarc_b200 import corpus

    c = corpus.c2_source_tree(total_bytes=600_000, seed=3)
    blob = corpus.materialise_host(emu, c)
    datas = [bytes(blob[int(o) : int(o) + int(l)]) for o, l in zip(c.off, c.len)]
    ours = sum(len(compress2(emu, d)) for d in datas)
    ref = sum(len(ref_path.ref_compress(d)) for d in datas)
    ratio_ours, ratio_ref = c.total_bytes / ours, c.total_bytes / ref
    print("ratio ours", ratio_ours, "ref L3", ratio_ref)
    assert ratio_ours > 0.85 * ratio_ref


def test_pack_batch_matches_reference_bookkeeping(emu):
    files = [text(3000, 1), rand(2000, 2), text(3000, 1), b"", text(200_000, 4), b"", rand(2000, 2), text(10, 9)]
    c = emu.zg_cctx_create()
    emu.check(emu.zg_cctx_init(c, 0))
    emu.check(emu.zg_cctx_set_parameter(c, 201, 1))
    emu.check(emu.zg_cctx_reset_archive(c, 12))
    r = pack_batch(emu, c, files)
    assert r["rc"] == 0
    # the reference path on the same ordered file list
    out = bytearray()
    enc = ref_path.RefEncoder(out, level=3)
    ref_digests = [enc.add_data_frame(f) for f in files]
    assert r["digests"] == ref_digests
    seen, first = set(), []
    for d in ref_digests:
        first.append(0 if d in seen else 1)
        seen.add(d)
    assert r["first"] == first
    # offsets: 12 + running sum of frame lengths in insertion order of unique contents
    pos = 12
    for i, f in enumerate(files):
        if first[i]:
            assert r["off"][i] == pos
            frame = r["frames"][pos - 12 : pos - 12 + r["len"][i]]
            _check_frame(emu, f, frame)
            pos += r["len"][i]
        else:
            j = ref_digests.index(ref_digests[i])
            assert (r["off"][i], r["len"][i]) == (r["off"][j], r["len"][j])
    assert pos - 12 == len(r["frames"]) and emu.zg_cctx_archive_offset(c) == pos
    # a second batch dedups against the first and continues the offsets
    files2 = [rand(2000, 2), text(777, 7), text(777, 7)]
    r2 = pack_batch(emu, c, files2)
    assert r2["first"] == [0, 1, 0]
    assert (r2["off"][0], r2["len"][0]) == (r["off"][1], r["len"][1])
    assert r2["off"][1] == pos and r2["off"][2] == pos
    _check_frame(emu, files2[1], r2["frames"])
    # our own decoder restores the whole archive too
    archive_frames = [r["frames"][o - 12 : o - 12 + l] for o, l, f1 in zip(r["off"], r["len"], first) if f1]
    uniq = [f for f, f1 in zip(files, first) if f1]
    outs, ok, status, rc = unpack_batch(emu, archive_frames, [len(f) for f in uniq], [d for d, f1 in zip(ref_digests, first) if f1])
    assert rc == 0 and outs == uniq and all(ok)
    emu.zg_cctx_free(c)


def test_pack_batch_capacity_error(emu):
    c = emu.zg_cctx_create()
    emu.check(emu.zg_cctx_reset_archive(c, 12))
    r = pack_batch(emu, c, [rand(5000, 3)], cap=100)
    assert emu.zg_get_error_code(r["rc"]) == 70
    emu.zg_cctx_free(c)


def test_sliced_host_api_and_chunked_encoder_equal_one_shot(emu):
    """zg_pack_batch/zg_unpack_batch cut a batch into double-buffered slices and the encoder cuts it into
    chunks: with tiny slice/chunk sizes (dedup pairs and a multi-block file straddling the cuts) the
    archive bytes, answers and restored files must equal the unsliced run."""
    import ctypes as C

    from zarc_b200 import corpus

    c = corpus.c2_source_tree(total_bytes=500_000, seed=11)
    blob = corpus.materialise_host(emu, c)
    files = [bytes(blob[int(o) : int(o) + int(l)]) for o, l in zip(c.off, c.len)]
    files += [files[1], files[0], bytes(blob[:150_000]) * 2, files[5], b"", b"x"]
    results = []
    try:
        for slice_bytes, chunk_bytes in ((0, 0), (70_000, 0), (0, 4096), (33_000, 65536)):
            emu.dll.zg_internal_set_slice_bytes(C.c_uint64(slice_bytes))
            emu.dll.zg_internal_set_encode_chunk_bytes(C.c_uint64(chunk_bytes))
            cctx = emu.zg_cctx_create()
            emu.check(emu.zg_cctx_init(cctx, 3))
            emu.check(emu.zg_cctx_set_parameter(cctx, 201, 1))
            emu.check(emu.zg_cctx_reset_archive(cctx, 12))
            r = pack_batch(emu, cctx, files)
            emu.zg_cctx_free(cctx)
            assert r["rc"] == 0
            frames = [bytes(r["frames"][o - 12 : o - 12 + l]) for o, l in zip(r["off"], r["len"])]
            outs, ok, status, rc = unpack_batch(emu, frames, [len(f) for f in files], r["digests"])
            assert rc == 0 and outs == files and all(ok)
            results.append((bytes(r["frames"]), r["digests"], r["first"], r["off"], r["len"]))
    finally:
        emu.dll.zg_internal_set_slice_bytes(C.c_uint64(0))
        emu.dll.zg_internal_set_encode_chunk_bytes(C.c_uint64(0))
    assert all(x == results[0] for x in results[1:])


@pytest.mark.parametrize("workers", [1, 2, 4])
def test_sliced_unpack_workers_and_frame_errors(emu, workers):
    """zg_unpack_batch decodes its slices with several contexts at once (host threads; the CPU test build runs them one
    after the other): whatever the worker count, every intact file comes back, a damaged frame is named in its own
    status entry, and the call's return code is the error of the FIRST damaged frame in batch order."""
    import ctypes as C

    files = [rand(3000 + 517 * i, 40 + i) + bytes(2000 + 10 * i) for i in range(40)]
    frames = [bytes(compress2(emu, f)) for f in files]
    digests = [ref_path.c_blake3(f) for f in files]
    try:
        emu.dll.zg_internal_set_slice_bytes(C.c_uint64(20_000))
        emu.dll.zg_internal_set_unpack_workers(C.c_int(workers))
        outs, ok, status, rc = unpack_batch(emu, frames, [len(f) for f in files], digests)
        assert rc == 0 and outs == files and all(ok) and not any(status)
        bad = list(frames)
        bad[31] = bad[31][:4] + bytes([bad[31][4] | 0x08]) + bad[31][5:]  # reserved bit of the frame header descriptor
        bad[7] = bad[7][:-4] + bytes(4)                                    # content checksum
        outs, ok, status, rc = unpack_batch(emu, bad, [len(f) for f in files], digests)
        assert emu.zg_get_error_code(rc) == 22  # checksum_wrong: frame 7 comes first
        assert status[7] == 22 and status[31] == 14 and [i for i, v in enumerate(status) if v] == [7, 31]
        assert all(o == f for i, (o, f) in enumerate(zip(outs, files)) if i not in (7, 31))
        assert [i for i, v in enumerate(ok) if not v] == [7, 31]
    finally:
        emu.dll.zg_internal_set_slice_bytes(C.c_uint64(0))
        emu.dll.zg_internal_set_unpack_workers(C.c_int(0))


def _pack_with(emu, files, level=3, params=()):
    cctx = emu.zg_cctx_create()
    emu.check(emu.zg_cctx_init(cctx, 0))
    emu.check(emu.zg_cctx_set_parameter(cctx, 201, 1))
    emu.check(emu.zg_cctx_set_parameter(cctx, 100, level))
    for p, v in params:
        emu.check(emu.zg_cctx_set_parameter(cctx, p, v))
    emu.check(emu.zg_cctx_reset_archive(cctx, 12))
    r = pack_batch(emu, cctx, files)
    emu.zg_cctx_free(cctx)
    assert r["rc"] == 0
    frames = [r["frames"][o - 12 : o - 12 + l] for o, l in zip(r["off"], r["len"])]
    for f, fr in zip(files, frames):
        assert ref_path.ref_decompress(fr, len(f)) == f  # whatever the parameters, libzstd restores the frames
        assert ref_path.ref_decompress_stream(bytes(fr), 0) == f
    return sum(len(fr) for fr in frames), frames


def test_levels_search_deeper_and_zstd_parameters_are_honoured_or_refused(emu):
    """Levels >= 6 / >= 9 keep 2 / 4 candidates per hash set; the --zstd parameters of pack.rs:140-195 either steer the
    match finder or are refused -- none is silently ignored."""
    from tests.golden.recipes import text

    rng = np.random.default_rng(11)
    words = [bytes(rng.integers(97, 123, int(rng.integers(3, 9)), dtype=np.uint8)) for _ in range(600)]
    src = b" ".join(words[int(i)] for i in rng.zipf(1.3, 60000) % 600)
    files = [src[:150_000], text(40_000, 3), src[150_000:230_000] + src[:20_000]]
    size = {lv: _pack_with(emu, files, level=lv)[0] for lv in (1, 3, 6, 9)}
    assert size[1] >= size[3] >= size[6] >= size[9] and size[9] < size[3]
    # searchLog / strategy reach the same search depths as the levels that imply them
    assert _pack_with(emu, files, 3, [(104, 2)])[0] == size[9]
    assert _pack_with(emu, files, 3, [(107, 7)])[0] == size[9]
    assert _pack_with(emu, files, 9, [(107, 1)])[0] == _pack_with(emu, files, 1)[0]  # strategy fast: greedy, one candidate
    # minMatch: no match shorter than asked for (and tests/test_encoder_edges_emu.py: repeats one byte too short stay
    # literals)
    from oracle import ref_path as rp

    for mm in (5, 7):
        total, frames = _pack_with(emu, files, 3, [(105, mm)])
        assert total > size[3]
        for f, fr in zip(files, frames):
            data, err, consumed, st = rp.c_zstd_decompress_frame(fr, len(f))
            assert err == 0 and st["sequences"] > 0 and st["min_match"] >= mm, (mm, st["min_match"])
    # windowLog below 16: no offset beyond the window (and tests/test_encoder_edges_emu.py: a repeat at exactly 2^w is
    # matched, at 2^w + 1 it is not); hashLog: a smaller table finds less
    total, frames = _pack_with(emu, files, 3, [(101, 10)])
    assert total > size[3]
    for f, fr in zip(files, frames):
        data, err, consumed, st = rp.c_zstd_decompress_frame(fr, len(f))
        assert err == 0 and st["sequences"] > 0 and st["max_offset"] <= 1 << 10, st["max_offset"]
    assert _pack_with(emu, files, 3, [(102, 8)])[0] > size[3]
    assert _pack_with(emu, files, 3, [(102, 20)])[0] == size[3]  # adjusted down to the largest table there is
    # refused: what has no counterpart
    cctx = emu.zg_cctx_create()
    for p, v, code in ((105, 3, 40), (103, 20, 40), (106, 64, 40), (105, 9, 42), (107, 12, 42), (101, 40, 42)):
        r = emu.zg_cctx_set_parameter(cctx, p, v)
        assert emu.zg_is_error(r) and emu.zg_get_error_code(r) == code, (p, v)
    for p in (103, 106):
        assert emu.zg_cctx_set_parameter(cctx, p, 0) == 0  # "not set" is fine
    emu.zg_cctx_free(cctx)

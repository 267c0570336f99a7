"""Pins the oracle (oracle/zarc_oracle.c + oracle/ref_path.py).

The reference has no tests or golden vectors for this path (SURVEY.md §8c), so the C restatement
is pinned against the same-version third-party libraries the reference links -- libzstd 1.5.5
(dlopen), Python blake3, xxhash -- and against the committed fixtures generated from them.
"""
import base64
import json
import os

import numpy as np
import pytest

from oracle import ref_path
from tests.golden.recipes import RECIPES, make_input, text, rand

HERE = os.path.dirname(os.path.abspath(__file__))
KAT = json.load(open(os.path.join(HERE, "golden", "kat.json")))


def test_libzstd_is_the_reference_version():
    assert ref_path.ZSTD_VERSION == 10505  # zstd-sys 2.0.9+zstd.1.5.5 (Cargo.lock:2480-2481)


def test_survey_known_answers():
    # SURVEY.md App. B / App. E
    assert ref_path.c_blake3(b"").hex() == "af1349b9f5f9a1a6a0404dea36dcc9499bcb25c9adc112b7cc9a93cae41f3262"
    assert ref_path.ref_compress(b"").hex() == "28b52ffd2400010000" + "99e9d851"
    assert ref_path.ref_compress(b"a").hex() == "28b52ffd2401090000" + "61" + "5b6e8ca9"
    assert ref_path.ref_compress(b"hello world\n").hex() == "28b52ffd240c610000" + b"hello world\n".hex() + "8c6d7d20"
    assert ref_path.ref_compress(bytes(1000)).hex() == "28b52ffd64e8024d000010000001" + "00e32b80055a074479"
    f = ref_path.ref_compress(b"hello zarc " * 1000)
    assert len(f) == 33 and f.hex().startswith("28b52ffd64f8299d000058") and f.hex().endswith("d269f6f1")


@pytest.mark.parametrize("case", KAT["cases"], ids=[c["recipe"] for c in KAT["cases"]])
def test_golden_vectors(case):
    import blake3
    import xxhash

    data = make_input(case["recipe"])
    assert len(data) == case["len"]
    # the fixture agrees with the live libraries ...
    assert blake3.blake3(data).hexdigest() == case["blake3"]
    assert f"{xxhash.xxh64(data, seed=0).intdigest():016x}" == case["xxh64"]
    # ... and the C restatement agrees with the fixture
    assert ref_path.c_blake3(data).hex() == case["blake3"]
    assert f"{ref_path.c_xxh64(data):016x}" == case["xxh64"]
    for level, b64 in case["frames"].items():
        frame = base64.b64decode(b64)
        assert ref_path.ref_compress(data, level=int(level)) == frame  # libzstd output is deterministic
        got, err, consumed, _ = ref_path.c_zstd_decompress_frame(frame, len(data))
        assert err == 0 and got == data and consumed == len(frame)


def test_c_decoder_vs_libzstd_feature_coverage():
    """The C decoder restores libzstd frames of levels 1/3/9 and the inputs exercise every section type
    the survey saw in reference-made frames (App. E)."""
    rng = np.random.default_rng(5)
    inputs = [make_input(n) for n in RECIPES]
    inputs += [text(400_000, 21), text(120_000, 22) + rand(140_000, 23) + text(200_000, 22)]
    inputs += [rng.integers(0, 4, 50_000, dtype=np.uint8).tobytes()]
    # fixed-shape records: every sequence has the same LL/ML/OF code -> RLE sequence tables
    inputs += [b"".join(b"RECORD_" + bytes([v]) for v in range(255))]
    seen = {}
    for data in inputs:
        for level in (1, 3, 9, 19):
            frame = ref_path.ref_compress(data, level=level)
            got, err, consumed, st = ref_path.c_zstd_decompress_frame(frame, len(data))
            assert err == 0, (len(data), level, err)
            assert got == data and consumed == len(frame)
            for k, v in st.items():
                seen[k] = seen.get(k, 0) + v
    for k in ("blocks_raw", "blocks_compressed", "lit_raw", "lit_huf1", "lit_huf4", "lit_treeless", "seq_predefined",
              "seq_fse", "seq_repeat", "seq_rle", "rep_offsets"):
        assert seen[k] > 0, k


def test_c_decoder_rejects_corruption():
    data = text(5000, 3)
    frame = bytearray(ref_path.ref_compress(data))
    frame[-1] ^= 1  # checksum
    _, err, _, _ = ref_path.c_zstd_decompress_frame(bytes(frame), len(data))
    assert err == 22
    _, err, _, _ = ref_path.c_zstd_decompress_frame(b"\x00" * 16, 16)
    assert err == 10
    good = ref_path.ref_compress(data)
    _, err, _, _ = ref_path.c_zstd_decompress_frame(good, len(data) - 1)
    assert err == 70
    _, err, _, _ = ref_path.c_zstd_decompress_frame(good[:-5], len(data))
    assert err != 0


def test_reference_call_sequence_dedup_and_offsets():
    """RefEncoder restates add_data_frame's bookkeeping (content_frame.rs:20-60)."""
    out = bytearray()
    enc = ref_path.RefEncoder(out, level=3)
    a, b = text(3000, 1), rand(2000, 2)
    da, db, da2 = enc.add_data_frame(a), enc.add_data_frame(b), enc.add_data_frame(a)
    assert da == da2 and da != db and len(enc.frames) == 2
    fa, fb = enc.frames[da], enc.frames[db]
    assert fa.offset == 12 and fb.offset == 12 + fa.length and len(out) == fb.offset + fb.length
    dec = ref_path.RefDecoder(bytes(out), enc.frames)
    assert dec.read_content_frame(da) == (a, True)
    assert dec.read_content_frame(db) == (b, True)
    assert dec.read_content_frame(b"\x00" * 32) is None


def _walk_headers(frame):
    """the section headers of a frame read directly (no entropy decoding): what the oracle's new statistics count"""
    desc = frame[4]
    fcs_flag, single, did = desc >> 6, (desc >> 5) & 1, desc & 3
    fcs_len = (1 if single else 0) if fcs_flag == 0 else (2, 4, 8)[fcs_flag - 1]
    p = 5 + (0 if single else 1) + (0, 1, 2, 4)[did] + fcs_len
    w = dict(fcs_size=fcs_len, blocks=0, lit={}, regen={}, nseq=[0, 0, 0], modes={}, trees={"direct": 0, "fse": 0})
    while True:
        bh = int.from_bytes(frame[p : p + 3], "little")
        last, btype, bsize = bh & 1, (bh >> 1) & 3, bh >> 3
        p += 3
        w["blocks"] += 1
        if btype == 2:
            q = p
            lt, sf = frame[q] & 3, (frame[q] >> 2) & 3
            if lt < 2:
                hb = {0: 1, 2: 1, 1: 2, 3: 3}[sf]
                regen = int.from_bytes(frame[q : q + hb], "little") >> (3 if hb == 1 else 4)
                q += hb + (regen if lt == 0 else 1)
            else:
                hb = {0: 3, 1: 3, 2: 4, 3: 5}[sf]
                v = int.from_bytes(frame[q : q + hb], "little")
                bits = {3: 10, 4: 14, 5: 18}[hb]
                regen, comp = (v >> 4) & ((1 << bits) - 1), v >> (4 + bits)
                if lt == 2:
                    w["trees"]["direct" if frame[q + hb] >= 128 else "fse"] += 1
                q += hb + comp
            w["lit"][(lt, sf)] = w["lit"].get((lt, sf), 0) + 1
            lo, hi = w["regen"].get(lt, (regen, regen))
            w["regen"][lt] = (min(lo, regen), max(hi, regen))
            b0 = frame[q]
            nseq = b0 if b0 < 128 else ((b0 - 128) << 8) + frame[q + 1] if b0 < 255 else frame[q + 1] + (frame[q + 2] << 8) + 0x7F00
            w["nseq"][0 if b0 < 128 else 1 if b0 < 255 else 2] += 1
            if nseq:
                m = frame[q + (1 if b0 < 128 else 2 if b0 < 255 else 3)]
                for t, sh in (("ll", 6), ("of", 4), ("ml", 2)):
                    key = (t, ref_path.SEQ_MODES[(m >> sh) & 3])
                    w["modes"][key] = w["modes"].get(key, 0) + 1
        p += 1 if btype == 1 else bsize
        if last:
            return w


def test_c_decoder_coverage_statistics_on_a_level19_frame():
    """The statistics the encoder edge cases rely on (oracle/zarc_oracle.c), on a libzstd level-19 frame of the inputs
    above: the header-level counts equal the frame's headers read directly, the sequence extremes agree with each
    other, and the blocks of a libzstd frame do read back into earlier blocks."""
    from tests.encoder_edge_cases import unique

    data = text(400_000, 21) + rand(140_000, 23) + text(200_000, 22) + unique(70_000, 5) + bytes(70_000)
    frame = ref_path.ref_compress(data, level=19)
    got, err, _, st = ref_path.c_zstd_decompress_frame(frame, len(data))
    assert err == 0 and got == data
    w = _walk_headers(frame)
    assert st["fcs_size"] == w["fcs_size"] == 4 and st["blocks"] == w["blocks"] == st["blocks_raw"] + st["blocks_rle"] + st["blocks_compressed"]
    for lt, kind in enumerate(ref_path.LIT_TYPES):
        for sf in range(4):
            assert st[f"lit_{kind}_sf{sf}"] == w["lit"].get((lt, sf), 0), (kind, sf)
        lo, hi = w["regen"].get(lt, (ref_path.NONE_SEEN, 0))
        assert (st[f"regen_min_{kind}"], st[f"regen_max_{kind}"]) == (lo, hi), kind
    assert st["huf_wdirect"] == w["trees"]["direct"] and st["huf_wfse"] == w["trees"]["fse"] and 5 <= st["huf_max_bits"] <= 11
    assert [st["nseq_h1"], st["nseq_h2"], st["nseq_h3"]] == w["nseq"]
    for t in ref_path.SEQ_TABLES:
        for m in ref_path.SEQ_MODES:
            assert st[f"{t}_{m}"] == w["modes"].get((t, m), 0), (t, m)
        assert sum(st[f"{t}_{m}"] for m in ref_path.SEQ_MODES) == sum(st[f"seq_{m}"] for m in ref_path.SEQ_MODES) // 3
    assert st["max_ll_log"] == 9 and st["max_ml_log"] == 9 and st["max_of_log"] >= 7  # level 19 uses the largest tables
    # the extremes: the 70 000 unmatchable bytes are one literal run (LL code 35), the zero run one long match (ML 52)
    assert st["max_lit_run"] >= 65_536 and st["max_ll_code"] == 35
    assert st["max_match"] >= 65_539 and st["max_ml_code"] == 52 and st["min_match"] >= 3
    assert st["max_offset"] > 131_072 and st["max_of_code"] >= 17  # (offBase = offset + 3 when not a repeat code)
    assert st["xblock_matches"] > 0  # the second copy of the text reaches back across blocks
    one = ref_path.ref_compress(text(100_000, 3), level=3)  # one block
    st1 = ref_path.c_zstd_decompress_frame(one, 100_000)[3]
    assert st1["blocks"] == 1 and st1["xblock_matches"] == 0 and st1["xblock_reps"] == 0


def test_c_decoder_counts_header_forms_and_cross_block_repeat_codes():
    """Statistics behind the encoder edge cases, on frames whose answer is known: a count below 128 written in the 2-byte
    Number_of_Sequences form is counted as 2 bytes (the form the frame used, not the smallest one for the count), and
    a repeat code that resolves to an offset set in the block before counts as a cross-block reference, while one that
    resolves to an initial repeat offset in the first block does not."""
    from tests import handmade_cases as H
    from tests import zstd_writer as W

    desc = H.frame(H.comp(H.raw_lit(b"abcdefgh"), [(2, 1, 4), W.seq(6, 3, 5)]),  # rep0 = 1 (initial), then offset 3
                   H.comp(H.raw_lit(b"xy"), [(2, 1, 4), W.seq(0, 7, 4)], nseq_form=2))  # rep0 = 3 from block 0
    frame, data = W.write(desc), W.execute(desc)
    got, err, _, st = ref_path.c_zstd_decompress_frame(frame, len(data))
    assert err == 0 and got == data == ref_path.ref_decompress(frame, len(data))
    assert (st["nseq_h1"], st["nseq_h2"], st["nseq_h3"]) == (1, 1, 0)
    assert st["blocks"] == 2 and st["rep_offsets"] == 2 and st["xblock_reps"] == 1 and st["xblock_matches"] == 2
    # libzstd carries repeat offsets across blocks of fixed-shape records
    data = b"".join(b"RECORD_" + bytes([v % 251]) for v in range(60_000))
    st = ref_path.c_zstd_decompress_frame(ref_path.ref_compress(data, level=3), len(data))[3]
    assert st["blocks"] > 1 and st["xblock_reps"] > 0

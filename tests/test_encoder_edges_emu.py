"""Encoder edge cases (tests/encoder_edge_cases.py) on the SIMT-emulator build, the parameters that steer the match
finder checked on the statistics of the frames, and the rare-path builds: the same sources with the tuning constants
that decide how often a rare path runs turned so that it runs nearly always."""
import pytest

from oracle import ref_path
from tests import encoder_edge_cases as E
from tests import handmade_cases as H
from tests.test_encode_emu import few_sequence_inputs
from tests.golden.recipes import text
from tests.test_hash_emu import SIZES, _data
from tests.helpers import unpack_batch, xxh64_batch


@pytest.mark.parametrize("name", list(E.CASES))
def test_encoder_edge(emu, name):
    E.run_case(emu, name)


@pytest.mark.parametrize("mm", [5, 6, 7])
def test_min_match_is_honoured(emu, mm):
    """minMatch: no match shorter than asked for; repeats of exactly mm - 1 bytes are matched by default and not at mm"""
    datas = [E.with_sequences(200, 300 + mm, ml=(mm - 1, mm)), text(100_000, 5)]
    st = E.check_frames(emu, datas, E.pack_frames(emu, datas, 3))
    assert st[0]["sequences"] >= 190 and st[0]["max_match"] == mm - 1  # the repeats are there, exactly mm - 1 long
    for level in (1, 3, 9):
        st = E.check_frames(emu, datas, E.pack_frames(emu, datas, level, [(105, mm)]))
        assert st[0]["sequences"] == 0, (level, st[0]["sequences"])
        assert st[1]["sequences"] > 0 and st[1]["min_match"] >= mm, (level, st[1]["min_match"])


@pytest.mark.parametrize("w", [10, 11, 12, 13, 14, 15])
def test_window_log_limits_the_distance(emu, w):
    """windowLog below 16: no offset beyond 2^w; a repeat at distance exactly 2^w is matched, one at 2^w + 1 is not"""
    phrase = E.unique(64, 7)
    at = lambda d: phrase + b"\x00" * (d - 64) + phrase  # noqa: E731
    datas = [at(1 << w), at((1 << w) + 1), text(100_000, 5)]
    for level in (1, 3, 9):
        st = E.check_frames(emu, datas, E.pack_frames(emu, datas, level, [(101, w)]))
        assert st[0]["max_offset"] == 1 << w, (level, st[0]["max_offset"])
        assert st[1]["max_offset"] == 1 and st[1]["regen_max_raw"] + st[1]["regen_max_huf"] >= 128, level
        assert all(s["max_offset"] <= 1 << w for s in st), level


# ---------------------------------------------------------------------------------------------------------------------
# rare-path builds: one module-scoped fixture per build (a build takes about 5 s of g++ and is cached under
# build/variants/).  Measured on 8 cores: the whole file takes about 3 minutes, the decoder-variant test 75 s of it
# (every sequence reconverges the emulated warp) and each chain variant 15 s (every case re-packed at three levels).
def _variant(defines):
    from zarc_b200 import _lib, build

    return _lib.Lib(build.build_emu_variant(defines), strict=False)


@pytest.fixture(scope="module", params=[["ZE_CHAIN_WARM=0u"], ["ZE_CHAIN_AHEAD=1"], ["ZE_CHAIN_AHEAD=3"]], ids=lambda d: " ".join(d))
def chain_variant(request):
    return _variant(request.param)


@pytest.fixture(scope="module")
def lane_cap_variant():
    return _variant(["ZE_LANE_CAP=8u"])


@pytest.fixture(scope="module")
def largest_logs_variant():
    return _variant(["ZE_LL_LOGCAP=9", "ZE_ML_LOGCAP=9", "ZE_OF_LOGCAP=8"])


@pytest.fixture(scope="module")
def whole_warp_copies_variant():
    return _variant(["ZD_LANE_COPY_MAX=1u", "ZD_B_STEPS=1"])


@pytest.fixture(scope="module")
def xxh64_warp_variant():
    return _variant(["XX_WARP_MIN=64u"])


def _all_frames(lib, levels=E.LEVELS):
    """every edge case's frames and the few-sequence inputs' frames, per level"""
    out = []
    for name in E.CASES:
        datas, _ = E.case_inputs(name)
        out += [E.pack_frames(lib, datas, lv) for lv in levels]
    few = few_sequence_inputs()
    out += [E.pack_frames(lib, few, lv) for lv in levels]
    return out


@pytest.fixture(scope="module")
def default_frames(emu):
    return _all_frames(emu)


def test_chain_variants_are_bit_identical(default_frames, chain_variant):
    """the FSE chain fields are those of the serial walk whatever the warm-up and look-ahead: with ZE_CHAIN_WARM=0 every
    lane below the first starts from a guessed state and re-walks its range when the guess was wrong"""
    assert _all_frames(chain_variant) == default_frames


def test_lane_cap_variant_frames_are_valid(lane_cap_variant):
    """ZE_LANE_CAP=8: nearly every match is extended by the whole warp.  The lazy rule compares lane-capped lengths, so
    the parse differs from the default's; the frames must still restore exactly"""
    for name in E.CASES:
        datas, _ = E.case_inputs(name)
        for lv in E.LEVELS:
            E.check_frames(lane_cap_variant, datas, E.pack_frames(lane_cap_variant, datas, lv), (name, lv))


def test_largest_table_logs_variant(largest_logs_variant):
    """FSE tables at the format's largest logs (9 / 9 / 8): valid frames, our decoder restores them, and log 9 was
    written"""
    lib = largest_logs_variant
    top = {"max_ll_log": 0, "max_ml_log": 0, "max_of_log": 0}
    for name in ("chain_ranges", "table_modes", "nseq_headers", "huf_limit"):
        datas, _ = E.case_inputs(name)
        for lv in E.LEVELS:
            for s in E.check_frames(lib, datas, E.pack_frames(lib, datas, lv), (name, lv)):
                for k in top:
                    top[k] = max(top[k], s[k])
    assert top["max_ll_log"] == 9 and top["max_ml_log"] == 9 and top["max_of_log"] >= 6, top


def test_decoder_whole_warp_copies_variant(whole_warp_copies_variant):
    """ZD_LANE_COPY_MAX=1, ZD_B_STEPS=1: every literal run and match copied by the whole warp, the warp reconverging after
    every sequence; exact restores of our frames (levels 1/3/9), libzstd's (1/3/9/19) and the hand-built ones"""
    lib = whole_warp_copies_variant
    for name in E.CASES:
        datas, _ = E.case_inputs(name)
        frames = [f for lv in E.LEVELS for f in E.pack_frames(lib, datas, lv)]
        frames += [ref_path.ref_compress(d, level=lv) for lv in (1, 3, 9, 19) for d in datas]
        want = datas * (len(frames) // len(datas))
        outs, ok, status, rc = unpack_batch(lib, frames, [len(d) for d in want], [ref_path.c_blake3(d) for d in want])
        assert rc == 0 and all(ok) and outs == want, (name, status)
    r = H.handmade_frames(lib, 0, 0)
    assert r["valid"] >= 140 and r["invalid"] >= 18


def test_xxh64_warp_path_variant(xxh64_warp_variant):
    """XX_WARP_MIN=64: every checksum of 64 bytes and more on the warp path, with every tail length"""
    import xxhash

    lib = xxh64_warp_variant
    files = [_data(n, 3) for n in SIZES] + [_data(64 + t, 9) for t in range(40)]
    for shift in (0, 1, 8):
        assert xxh64_batch(lib, files, shift=shift) == [xxhash.xxh64(f, seed=0).intdigest() for f in files], shift
    datas, _ = E.case_inputs("blocks")
    E.check_frames(lib, datas, E.pack_frames(lib, datas, 3))  # checksums made and verified on this path

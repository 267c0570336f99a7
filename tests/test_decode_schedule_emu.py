"""The decoder's scheduling layer (tests/decode_schedule_cases.py) on the SIMT-emulator build: sequence-arena deferrals,
hand-out settings from 2 to 32 frames a batch, and the rounds of the Huffman literals pre-pass at their edges.  Bytes,
statuses and return codes must not change with any of them; the emulator's counters must equal the arithmetic that
says which deferrals and rounds each case reaches.  The same on a build with a 4160-entry table space and groups of
5 sections (a group size that does not divide 32)."""
import pytest

from tests import decode_schedule_cases as S

# deferred set-ups at 32 frames a batch, by the arithmetic of decode_schedule_cases.arena_defers
DEFERS_AT_32 = {"arena_full": 0, "arena_full_plus_one": 1, "arena_bad_literals_deferred": 1, "max_seq_three_a_round": 7,
                "arena_mixed": 3, "arena_mixed_reversed": 4}
# pre-pass rounds of the default build (8192 entries, groups of 32), by the arithmetic of prepass_rounds
ROUNDS = {"bits11_x4_fills_the_table_space": 1, "bits11_x5": 2, "streams4_x8_fill_32_lanes": 1, "streams4_x9": 2,
          "streams4_x7_and_1_stream_x4": 1, "bits11_x2_and_6": 1, "bits11_x2_and_7": 1}
# ... and of the variant (4160 entries, groups of 5)
ROUNDS_4160_5 = {"bits11_x4_fills_the_table_space": 2, "bits11_x5": 3, "streams4_x8_fill_32_lanes": 2, "streams4_x9": 2,
                 "streams4_x7_and_1_stream_x4": 3, "bits11_x2_and_6": 1, "bits11_x2_and_7": 2}
VARIANT = ["ZD_HL_TAB=4160u", "ZD_HL_SECS=5u"]


@pytest.fixture(scope="module")
def variant():
    from zarc_b200 import _lib, build

    return _lib.Lib(build.build_emu_variant(VARIANT), strict=False)


def test_frames_agree_with_the_references_and_reach_the_edges():
    arena = S.arena_cases()
    for _, items in arena:
        S.check_reference(items)
    S.check_reference(S.lane_path_items())
    for _, secs in S.prepass_cases():
        S.check_reference(S.prepass_items(secs))
    # the arena arithmetic: exactly full, one past it, three of the largest blocks a round
    assert 4 * S.DENSE == S.ARENA and 3 * S.MAX_SEQ <= S.ARENA < 4 * S.MAX_SEQ
    for name, items in arena:
        assert S.arena_defers(items, 32) == DEFERS_AT_32[name], name
        assert S.arena_defers(items, 2) == 0, name
    assert S.arena_defers(S.lane_path_items(), 32) == 4
    # the pre-pass arithmetic: 4 x 2048 = 8192 entries, 8 x 4 = 7 x 4 + 4 = 32 streams, 2 x 2048 + 64 = 4160
    cases = dict(S.prepass_cases())
    assert [s.bits for s in cases["bits11_x4_fills_the_table_space"]] == [11] * 4
    assert [s.bits for s in cases["bits11_x2_and_6"]] == [11, 11, 6] and cases["bits11_x2_and_7"][2].bits == 7
    assert sum(s.streams for s in cases["streams4_x7_and_1_stream_x4"]) == 32
    for name, secs in cases.items():
        if name.startswith("bad_"):
            assert sum(s.streams for s in secs) == 32, name
        assert S.prepass_rounds(secs, 8192, 32) == ROUNDS.get(name, 1), name  # (a bad section's case: one full round)
        if name in ROUNDS_4160_5:
            assert S.prepass_rounds(secs, 4160, 5) == ROUNDS_4160_5[name], name


@pytest.mark.parametrize("name", list(DEFERS_AT_32))
def test_arena_cases_every_hand_out(emu, name):
    items = dict(S.arena_cases())[name]
    assert S.check_arena_case(emu, name, items) == DEFERS_AT_32[name]


def test_deferred_blocks_of_multi_block_frames_on_the_lane_path(emu):
    """Treeless literals, Repeat_Mode tables, repeat offsets and the Raw / RLE blocks before it: what a block deferred
    a round keeps; then the same batch on the default path"""
    items = S.lane_path_items()
    assert S.check_arena_case(emu, "lane_path", items, lane_path=True) == 4
    S.run_batch(emu, items, "default path")


def test_mixed_batch_every_hand_out(emu):
    pool = S.mixed_pool(emu)
    for count in S.MIXED_COUNTS:
        S.run_settings(emu, S.mixed_batch(pool, count), ("mixed", count))


@pytest.mark.parametrize("name", [n for n, _ in S.prepass_cases()])
def test_prepass_rounds(emu, name):
    secs = dict(S.prepass_cases())[name]
    S.sched_stats(emu)
    S.run_batch(emu, S.prepass_items(secs), name)
    assert S.sched_stats(emu)[1] == S.prepass_rounds(secs, 8192, 32), name


def test_variant_4160_entries_groups_of_5(variant):
    for name, secs in S.prepass_cases():
        S.sched_stats(variant)
        S.run_batch(variant, S.prepass_items(secs), name)
        assert S.sched_stats(variant)[1] == S.prepass_rounds(secs, 4160, 5), name
    for name, items in S.arena_cases():
        if name != "max_seq_three_a_round":  # (the slowest on the emulator; the default build runs it)
            assert S.check_arena_case(variant, name, items) == DEFERS_AT_32[name]
    assert S.check_arena_case(variant, "lane_path", S.lane_path_items(), lane_path=True) == 4
    pool = S.mixed_pool(variant)
    for count in (33, 65):
        S.run_batch(variant, S.mixed_batch(pool, count), ("mixed", count))

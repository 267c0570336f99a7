"""The decoder's scheduling layer (tests/decode_schedule_cases.py) on the GPU: the arena, lane-path, mixed-batch and
pre-pass cases under every hand-out setting, a scale run of about a thousand sequence-dense frames among a C2-shaped
batch, and the product built with a 4160-entry table space and groups of 5 pre-pass sections.  The product has no
scheduling counters: which deferrals and rounds each case reaches is the arithmetic the CPU suite checks against the
emulator's counters (tests/test_decode_schedule_emu.py)."""
import pytest

from tests import decode_schedule_cases as S

pytestmark = pytest.mark.gpu

VARIANT = ["ZD_HL_TAB=4160u", "ZD_HL_SECS=5u"]


@pytest.mark.parametrize("name", [n for n, _ in S.arena_cases(scale=4)])
def test_arena_cases_every_hand_out(gpu, name):
    items = dict(S.arena_cases(scale=4))[name]
    n = S.check_arena_case(gpu, name, items)
    assert n > 0 or name == "arena_full", (name, "no deferral at 32 frames a batch")


def test_deferred_blocks_of_multi_block_frames_on_the_lane_path(gpu):
    items = S.lane_path_items()
    assert S.check_arena_case(gpu, "lane_path", items, lane_path=True) == 4
    S.run_batch(gpu, items, "default path")


def test_mixed_batch_every_hand_out(gpu):
    pool = S.mixed_pool(gpu)
    for count in S.MIXED_COUNTS:
        S.run_settings(gpu, S.mixed_batch(pool, count), ("mixed", count))


def test_prepass_rounds(gpu):
    for name, secs in S.prepass_cases():
        S.run_batch(gpu, S.prepass_items(secs), name)


def test_scale_dense_frames_among_a_c2_batch(gpu):
    """1 000 sequence-dense frames (32 768 and 43 690 sequences) with a C2-shaped batch packed by libzstd (level 19) and
    by this encoder: byte-identical restores at 32 and at 2 frames a batch and at the defaults"""
    from oracle import ref_path
    from tests import encoder_edge_cases as E
    from zarc_b200 import corpus

    c = corpus.c2_source_tree(total_bytes=16_000_000, seed=31)
    blob = corpus.materialise_host(gpu, c)
    datas = [bytes(blob[int(o) : int(o) + int(n)]) for o, n in zip(c.off, c.len)]
    items = [S.Item(f"c2.zstd19.{i}", ref_path.ref_compress(d, level=19), d) for i, d in enumerate(datas)]
    items += [S.Item(f"c2.ours.{i}", f, d) for i, (d, f) in enumerate(zip(datas, E.pack_frames(gpu, datas, 3)))]
    dense = [S.dense("raw", 1), S.dense("huf", 2), S.dense("raw", 3), S.dense("huf", 4), S.max_seq(b"A"), S.max_seq(b"B")]
    batch = []
    for i in range(1000):  # dense frames spread through the batch
        batch.append(dense[i % len(dense)])
        batch += items[i * len(items) // 1000 : (i + 1) * len(items) // 1000]
    assert len(batch) == 1000 + len(items)
    S.run_settings(gpu, batch, "scale", settings=[s for s in S.SETTINGS if s[0] in ("want32", "want2", "defaults")])


def test_variant_4160_entries_groups_of_5(gpu):
    from zarc_b200 import _lib, build

    lib = _lib.Lib(build.build_product_variant(VARIANT), strict=False)
    assert lib.zg_build_info() == b"sm_100a"
    for name, secs in S.prepass_cases():
        S.run_batch(lib, S.prepass_items(secs), name)
    for name, items in S.arena_cases():
        S.check_arena_case(lib, name, items)
    assert S.check_arena_case(lib, "lane_path", S.lane_path_items(), lane_path=True) == 4
    pool = S.mixed_pool(lib)
    for count in S.MIXED_COUNTS:
        S.run_batch(lib, S.mixed_batch(pool, count), ("mixed", count))

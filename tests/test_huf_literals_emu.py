"""The Huffman literals pre-pass (k_zd_huf_literals) at one section per warp, on the SIMT-emulator build: every group is a
group of one, 1-stream sections take a single lane, and every section's tree and table go through the same shared-memory
slot.  The default build (two sections per warp, so a partial last group whenever the count is odd) runs through the
rest of the decoder tests."""
import pytest

from oracle import ref_path
from tests import encoder_edge_cases as E
from tests import handmade_cases as H
from tests.helpers import unpack_batch


@pytest.fixture(scope="module")
def one_section_variant():
    from zarc_b200 import _lib, build

    return _lib.Lib(build.build_emu_variant(["ZD_HL_SECS=1u"]), strict=False)


def test_one_section_per_warp_variant(one_section_variant):
    """exact restores of our frames (level 3), libzstd's (1/3/9/19) and the hand-built ones, valid and invalid"""
    lib = one_section_variant
    for name in ("raw_headers", "huf_headers", "huf_limit", "weights", "blocks"):
        datas, _ = E.case_inputs(name)
        frames = E.pack_frames(lib, datas, 3) + [ref_path.ref_compress(d, level=lv) for lv in (1, 3, 9, 19) for d in datas]
        want = datas * (len(frames) // len(datas))
        outs, ok, status, rc = unpack_batch(lib, frames, [len(d) for d in want], [ref_path.c_blake3(d) for d in want])
        assert rc == 0 and all(ok) and outs == want, (name, status)
    r = H.handmade_frames(lib, 0, 0)
    assert r["valid"] >= 140 and r["invalid"] >= 18

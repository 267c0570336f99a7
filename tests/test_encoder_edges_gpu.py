"""Encoder edge cases (tests/encoder_edge_cases.py) on the GPU, and the two rare-path builds whose paths are the
hardware's own: the FSE chain re-walk (ZE_CHAIN_WARM=0: frames bit-identical to the default build) and the whole-warp
copies of the decoder with the warp path of XXH64 for every checksum (ZD_LANE_COPY_MAX=1, XX_WARP_MIN=64: exact
restores), each also on a C2-shaped batch of a few MB.  A variant build is one nvcc run of the sources into
build/variants/."""
import pytest

from oracle import ref_path
from tests import encoder_edge_cases as E
from tests.helpers import unpack_batch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", list(E.CASES))
def test_encoder_edge(gpu, name):
    E.run_case(gpu, name)


def _variant(defines):
    from zarc_b200 import _lib, build

    lib = _lib.Lib(build.build_product_variant(defines), strict=False)
    assert lib.zg_build_info() == b"sm_100a"
    return lib


@pytest.fixture(scope="module")
def c2_batch(gpu):
    from zarc_b200 import corpus

    c = corpus.c2_source_tree(total_bytes=4_000_000, seed=21)
    blob = corpus.materialise_host(gpu, c)
    return [bytes(blob[int(o) : int(o) + int(n)]) for o, n in zip(c.off, c.len)]


def _frames(lib, datas_list, levels=E.LEVELS):
    return [E.pack_frames(lib, d, lv) for d in datas_list for lv in levels]


def test_chain_rewalk_variant_is_bit_identical(gpu, c2_batch):
    inputs = [E.case_inputs(n)[0] for n in E.CASES] + [c2_batch]
    assert _frames(_variant(["ZE_CHAIN_WARM=0u"]), inputs) == _frames(gpu, inputs)


def test_whole_warp_copies_and_xxh64_warp_variant(gpu, c2_batch):
    lib = _variant(["ZD_LANE_COPY_MAX=1u", "XX_WARP_MIN=64u"])
    for name in E.CASES:
        datas, _ = E.case_inputs(name)
        for lv in E.LEVELS:
            E.check_frames(lib, datas, E.pack_frames(gpu, datas, lv), (name, lv))
        frames = [ref_path.ref_compress(d, level=19) for d in datas]
        outs, ok, status, rc = unpack_batch(lib, frames, [len(d) for d in datas], [ref_path.c_blake3(d) for d in datas])
        assert rc == 0 and all(ok) and outs == datas, (name, status)
    frames = E.pack_frames(lib, c2_batch, 3)
    assert frames == E.pack_frames(gpu, c2_batch, 3)  # the encoder is untouched by these constants
    outs, ok, status, rc = unpack_batch(lib, frames, [len(d) for d in c2_batch], [ref_path.c_blake3(d) for d in c2_batch])
    assert rc == 0 and all(ok) and outs == c2_batch

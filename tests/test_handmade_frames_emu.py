"""Hand-built frames (tests/handmade_cases.py) on the SIMT-emulator build: the writer checked against libzstd and the
C oracle, then every decode path against the bytes the descriptions call for."""
import numpy as np

from tests import handmade_cases as H


def test_writer_agrees_with_libzstd_and_the_c_oracle():
    cases = H.valid_cases()
    for seed in range(3):
        rng = np.random.default_rng(1000 + seed)
        cases += [(f"seed{seed}.{i}", H.random_description(rng)) for i in range(8)]
    st = H.check_writer(cases)
    # the modes the catalogue is about were actually written
    for k in ("lit_treeless", "lit_huf1", "lit_huf4", "seq_rle", "seq_fse", "seq_repeat", "seq_predefined", "rep_offsets",
              "single_segment", "blocks_raw", "blocks_rle", "lit_raw", "lit_rle"):
        assert st[k] > 0, k


def test_named_frames_every_path(emu):
    r = H.handmade_frames(emu, 0, 0)
    assert r["valid"] >= 140 and r["invalid"] >= 18


def test_random_frames_every_path(emu):
    r = H.handmade_frames(emu, 1, 3, named=False)
    assert r["valid"] == 24

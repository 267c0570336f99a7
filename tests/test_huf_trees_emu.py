"""Huffman trees read one lane per section (k_zd_huf_literals) on the SIMT-emulator build: every edge of a tree
description, jump table and stream, bad sections in the same groups as good ones (tests/huf_tree_cases.py)."""
from tests import huf_tree_cases as T


def test_tree_edges_in_mixed_groups(emu):
    """exactly the bad sections fail, with ZSTD_error_corruption_detected; libzstd and the two-block path agree"""
    good, bad = T.check_cases(emu, 0)
    assert good >= 20 and bad >= 20


def test_tree_byte_mutations(emu):
    """whatever is accepted after changing tree-description bytes is what libzstd restores"""
    acc, rej = T.mutate_trees(emu, 1, rounds=3)
    assert acc > 0 and rej > 0

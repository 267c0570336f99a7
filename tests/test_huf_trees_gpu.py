"""Huffman trees read one lane per section (k_zd_huf_literals) on the GPU: the edge cases of tests/huf_tree_cases.py
and more tree-byte mutations than the CPU suite runs."""
import pytest

from tests import huf_tree_cases as T

pytestmark = pytest.mark.gpu


def test_tree_edges_in_mixed_groups(gpu):
    for seed in range(4):
        good, bad = T.check_cases(gpu, seed)
    assert good >= 20 and bad >= 20


def test_tree_byte_mutations(gpu):
    acc, rej = T.mutate_trees(gpu, 2, rounds=40)
    assert acc > 0 and rej > 0

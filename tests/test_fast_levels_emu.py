"""Negative compression levels (tests/fast_level_cases.py) on the SIMT-emulator build: a C2-shaped batch of about 2 MB
and the boundary inputs at levels -1 .. -131072."""
import numpy as np
import pytest

from tests import fast_level_cases as F


@pytest.fixture(scope="module")
def inputs(emu):
    c2 = F.c2_batch(emu, 2_000_000)
    return c2, c2 + F.edge_inputs()


def test_fast_levels(emu, inputs):
    c2, datas = inputs
    ours, ref, factors = F.run_levels(emu, datas, len(c2))
    print("ours", ours, "libzstd", ref, "factors", factors)


def test_fast_level_combinations(emu, inputs):
    F.check_combinations(emu, inputs[0][:40] + F.edge_inputs()[:6])


def test_fast_level_parameters_keep_their_meaning(emu, inputs):
    F.check_fast_parameters(emu, inputs[0][:40] + F.edge_inputs())


def test_fast_level_same_bytes_on_every_path(emu, inputs):
    # (the emulator's device memory is host memory: numpy buffers stand in for device buffers)
    F.check_paths(emu, inputs[0][:60] + F.edge_inputs(), to_dev=lambda a: (a, a.ctypes.data), to_host=np.asarray)

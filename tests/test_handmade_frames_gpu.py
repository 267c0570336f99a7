"""Hand-built frames (tests/handmade_cases.py) on the GPU: the named cases and more random descriptions than the CPU
suite runs, through every decode path."""
import pytest

from tests import handmade_cases as H

pytestmark = pytest.mark.gpu


def test_named_frames_every_path(gpu):
    r = H.handmade_frames(gpu, 0, 0)
    assert r["valid"] >= 140 and r["invalid"] >= 18


def test_random_frames_every_path(gpu):
    r = H.handmade_frames(gpu, 1, 40, named=False)
    assert r["valid"] == 320

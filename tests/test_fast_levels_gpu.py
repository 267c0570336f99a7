"""Negative compression levels (tests/fast_level_cases.py) on the GPU: the emulator's checks on a larger C2-shaped batch,
the CLI round trip of a small tree read back by the reference container reader, and a 256 MB batch at -1 and -5 packed
and unpacked on the device with its digests verified."""
import os
import subprocess

import numpy as np
import pytest

from tests import fast_level_cases as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def inputs(gpu):
    c2 = F.c2_batch(gpu, 16_000_000)
    return c2, c2 + F.edge_inputs()


def _to_dev(a):
    import torch

    t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).cuda()
    return t, t.data_ptr()


def _to_host(t):
    return t.cpu().numpy()


def test_fast_levels(gpu, inputs):
    c2, datas = inputs
    ours, ref, factors = F.run_levels(gpu, datas, len(c2))
    print("ours", ours, "libzstd", ref, "factors", factors)


def test_fast_level_combinations(gpu, inputs):
    F.check_combinations(gpu, inputs[0][:200] + F.edge_inputs()[:6])


def test_fast_level_parameters_keep_their_meaning(gpu, inputs):
    F.check_fast_parameters(gpu, inputs[0][:200] + F.edge_inputs())


def test_fast_level_same_bytes_on_every_path(gpu, inputs):
    F.check_paths(gpu, inputs[0][:400] + F.edge_inputs(), to_dev=_to_dev, to_host=_to_host)


def test_cli_pack_level_minus_5_round_trip(gpu, tmp_path):
    from oracle import ref_container, ref_path
    from tests import container_cases as cc
    from zarc_b200 import _lib

    (tmp_path / "tree").mkdir()
    files = cc.make_tree(str(tmp_path / "tree"))
    cc.run_cli(_lib.PRODUCT_SO, ["pack", "--level", "-5", "--output", str(tmp_path / "out.zarc"), "tree"], cwd=str(tmp_path))
    ar = ref_container.read_archive((tmp_path / "out.zarc").read_bytes())
    by_name = {"/".join(f[1]): f for f in ar["files"]}
    for rel, content in files.items():
        got, ok = ar["content"](by_name["tree/" + rel][2])
        assert got == content and ok and by_name["tree/" + rel][2] == ref_path._blake3(content), rel
    (tmp_path / "x").mkdir()
    cc.run_cli(_lib.PRODUCT_SO, ["unpack", str(tmp_path / "out.zarc")], cwd=str(tmp_path / "x"))
    for rel, content in files.items():
        assert (tmp_path / "x" / "tree" / rel).read_bytes() == content, rel


@pytest.mark.parametrize("level", [-1, -5])
def test_256mb_batch_round_trip(gpu, level):
    import torch

    from tests.test_big_frames_gpu import _pack_dev, _unpack_dev
    from zarc_b200 import corpus

    c = corpus.c2_source_tree(total_bytes=256_000_000, seed=13)
    so, sl, sk, key = c.segments()
    blob = torch.empty(max(c.blob_bytes, 1) + 64, dtype=torch.uint8, device="cuda")
    d = [torch.from_numpy(x).cuda() for x in (so, sl, sk, key)]
    gpu.check(gpu.zg_corpus_generate_dev(0, blob.data_ptr(), d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), len(so)))
    torch.cuda.synchronize()
    p = _pack_dev(gpu, torch, blob, c, level=level)
    assert p["nbytes"] < c.total_bytes
    rc, out, ok, st, _ = _unpack_dev(gpu, torch, p["frames"], p["foff"], p["flen"], p["len"], p["dig"], p["off"], c.blob_bytes)
    assert rc == 0 and all(ok) and not any(st)
    assert torch.equal(out[: c.blob_bytes], blob[: c.blob_bytes])

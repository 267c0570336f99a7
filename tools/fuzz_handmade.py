"""Long run of the hand-built frame checks (tests/handmade_cases.py): random frame descriptions through every decode
path, each compared with the bytes the description calls for.
    python tools/fuzz_handmade.py [--emu] [--first N] [--count N]"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tests import handmade_cases  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--emu", action="store_true", help="the SIMT-emulator build instead of the GPU library")
    ap.add_argument("--first", type=int, default=100_000)
    ap.add_argument("--count", type=int, default=500)
    a = ap.parse_args()
    from zarc_b200 import _lib, build

    lib = _lib.Lib(build.build_emu(), strict=False) if a.emu else _lib.lib()
    t0 = time.time()
    r = handmade_cases.handmade_frames(lib, a.first, a.count, log=lambda s, n: print(f"seed {s}: {n} frames, {time.time() - t0:.0f} s", flush=True))
    print(f"handmade frames: {r['valid']} valid frames restored on every path, {r['invalid']} invalid ones rejected "
          f"(seeds {a.first}..{a.first + a.count - 1}, {time.time() - t0:.0f} s)")


if __name__ == "__main__":
    main()

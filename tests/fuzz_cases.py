"""Randomised checks shared by the CPU test-suite (a few seeds each, tests/test_fuzz_emu.py) and by the longer runs of
tools/fuzz_*.py (thousands of seeds; results in profiles/README.md).  Every function takes the library to test (the
SIMT-emulator build on the CPU, the product library on a GPU) and a range of seeds, raises AssertionError on the first
disagreement with the reference path (oracle/ref_path.py: libzstd 1.5.5 + BLAKE3 called the way the reference calls them)
and returns counters."""
import ctypes as C
import os
import shutil
import struct
import subprocess
import tempfile

import numpy as np

from oracle import ref_container, ref_path
from tests.golden.recipes import rand, text
from tests.helpers import compress2, pack_batch, unpack_batch


def glued_input(rng, scale=1.0, max_parts=6, sizes=(0, 1, 3, 7, 31, 100, 1000, 5000, 40000, 131072, 200000)):
    """random / text / runs / periodic / noisy text / copies of earlier parts, glued"""
    parts = []
    for _ in range(int(rng.integers(0, max_parts))):
        k = int(rng.integers(0, 6))
        m = int(int(rng.choice(sizes)) * scale) + int(rng.integers(0, 64))
        if k == 0:
            parts.append(rand(m, int(rng.integers(1, 1 << 30))))
        elif k == 1:
            parts.append(text(m, int(rng.integers(1, 1 << 30))))
        elif k == 2:
            parts.append(bytes([int(rng.integers(0, 256))]) * m)
        elif k == 3 and parts:
            parts.append(parts[int(rng.integers(0, len(parts)))][:m])
        elif k == 4:
            unit = rand(int(rng.integers(1, 40)), int(rng.integers(1, 1 << 30)))
            parts.append((unit * (m // max(1, len(unit)) + 1))[:m])
        else:
            a = bytearray(text(m, 77))
            for _ in range(m // 50):
                if m:
                    a[int(rng.integers(0, m))] = int(rng.integers(0, 256))
            parts.append(bytes(a))
    return b"".join(parts)


def encode_roundtrips(lib, first, count, levels=(1, 3, 6, 9), log=None):
    """Frames made by this library's encoder: restored byte-identically by libzstd and by our decoder, digests verified;
    every block independent of the blocks before it (no match reaches into one, no repeat code resolves to an offset set
    in one: the C oracle's statistics)."""
    frames_done = 0
    for seed in range(first, first + count):
        rng = np.random.default_rng(seed)
        datas = [glued_input(rng) for _ in range(6)]
        for level in levels:
            frames = []
            for d in datas:
                fr = bytes(compress2(lib, d, level=level, checksum=bool(rng.integers(0, 2))))
                assert ref_path.ref_decompress(fr, len(d)) == d, (seed, level, len(d), "libzstd restores something else")
                got, err, _, st = ref_path.c_zstd_decompress_frame(fr, len(d))
                assert err == 0 and got == d, (seed, level, len(d), "the C oracle restores something else", err)
                assert st["xblock_matches"] == 0 and st["xblock_reps"] == 0, (seed, level, len(d), "a block depends on an earlier one")
                frames.append(fr)
            outs, ok, status, rc = unpack_batch(lib, frames, [len(d) for d in datas], [ref_path.c_blake3(d) for d in datas])
            assert rc == 0 and outs == datas and all(ok), (seed, level, rc, status)
            frames_done += len(frames)
        if log and seed % 5 == 0:
            log(seed, frames_done)
    return frames_done


def decode_reference_frames(lib, first, count, levels=(1, 3, 9, 19), log=None):
    """Frames made by libzstd the way the reference makes them (multi-block, blocks reading earlier blocks, Repeat_Mode
    tables, Treeless literals, RLE blocks): restored byte-identically by our decoder, digests verified."""
    frames_done = 0
    for seed in range(first, first + count):
        rng = np.random.default_rng(seed)
        datas = [glued_input(rng, float(rng.choice([0.1, 1.0, 1.0, 2.0])), 8, (0, 1, 7, 100, 1000, 5000, 40000, 131072, 200000, 500000)) for _ in range(5)]
        for level in levels:
            frames = [ref_path.ref_compress(d, level=level, checksum=bool(rng.integers(0, 2))) for d in datas]
            outs, ok, status, rc = unpack_batch(lib, frames, [len(d) for d in datas], [ref_path.c_blake3(d) for d in datas])
            assert rc == 0 and outs == datas and all(ok), (seed, level, rc, status, [len(d) for d in datas])
            frames_done += len(frames)
        if log and seed % 5 == 0:
            log(seed, frames_done)
    return frames_done


def _pack_file(rng):
    k = int(rng.integers(0, 5))
    m = int(rng.choice([0, 0, 1, 50, 700, 3000, 20000, 131072, 140000, 300000])) + int(rng.integers(0, 16))
    if m <= 16 and rng.integers(0, 2):
        m = 0
    s = int(rng.integers(1, 1 << 30))
    if k == 0:
        return rand(m, s)
    if k == 1:
        return bytes([s & 255]) * m
    return text(m, s)


def pack_bookkeeping(lib, first, count, log=None):
    """Random file lists with duplicates (within and across batches), empty and multi-block files, packed in a random
    number of zg_pack_batch calls under random host-API slice and encoder chunk sizes: digests, first-occurrence flags,
    offsets and lengths equal the reference Encoder's bookkeeping (content_frame.rs:20-60: offsets 12 + running sum in
    insertion order of unique contents, a duplicate answers with its first occurrence's frame), the archive bytes do not
    depend on how the work was cut, every frame is restored by libzstd and by our decoder."""
    try:
        for seed in range(first, first + count):
            rng = np.random.default_rng(seed)
            pool = [_pack_file(rng) for _ in range(int(rng.integers(1, 12)))]
            files = [pool[int(rng.integers(0, len(pool)))] for _ in range(int(rng.integers(1, 30)))]
            level = int(rng.choice([1, 3, 9]))
            enc = ref_path.RefEncoder(bytearray(), level=level)
            ref_digests = [enc.add_data_frame(f) for f in files]
            seen, first_flags = {}, []
            for i, d in enumerate(ref_digests):
                first_flags.append(0 if d in seen else 1)
                seen.setdefault(d, i)
            archives = []
            for _trial in range(2):
                lib.dll.zg_internal_set_slice_bytes(C.c_uint64(int(rng.choice([0, 10_000, 70_000, 400_000]))))
                lib.dll.zg_internal_set_encode_chunk_bytes(C.c_uint64(int(rng.choice([0, 4096, 65536, 262144]))))
                cuts = sorted(set(int(x) for x in rng.integers(0, len(files) + 1, int(rng.integers(0, 3))))) + [len(files)]
                c = lib.zg_cctx_create()
                lib.check(lib.zg_cctx_init(c, 0))
                lib.check(lib.zg_cctx_set_parameter(c, 201, 1))
                lib.check(lib.zg_cctx_set_parameter(c, 100, level))
                lib.check(lib.zg_cctx_reset_archive(c, 12))
                got = dict(digests=[], first=[], off=[], len=[], frames=b"")
                a = 0
                for b in cuts:
                    r = pack_batch(lib, c, files[a:b])
                    assert r["rc"] == 0, (seed, r["rc"])
                    for k in ("digests", "first", "off", "len"):
                        got[k] += r[k]
                    got["frames"] += r["frames"]
                    a = b
                assert lib.zg_cctx_archive_offset(c) == 12 + len(got["frames"])
                lib.zg_cctx_free(c)
                assert got["digests"] == ref_digests, seed
                assert got["first"] == first_flags, seed
                pos = 12
                for i in range(len(files)):
                    if first_flags[i]:
                        assert got["off"][i] == pos, (seed, i)
                        pos += got["len"][i]
                    else:
                        j = seen[ref_digests[i]]
                        assert (got["off"][i], got["len"][i]) == (got["off"][j], got["len"][j]), (seed, i)
                assert pos - 12 == len(got["frames"])
                archives.append(got["frames"])
            assert archives[0] == archives[1], (seed, "archive bytes depend on slices / chunks / batch cuts")
            fr = [got["frames"][o - 12 : o - 12 + l] for o, l, f1 in zip(got["off"], got["len"], first_flags) if f1]
            uniq = [f for f, f1 in zip(files, first_flags) if f1]
            for f, x in zip(uniq, fr):
                assert ref_path.ref_decompress(x, len(f)) == f, seed
            outs, ok, status, rc = unpack_batch(lib, fr, [len(f) for f in uniq], [d for d, f1 in zip(ref_digests, first_flags) if f1])
            assert rc == 0 and outs == uniq and all(ok), seed
            if log and seed % 10 == 0:
                log(seed, seed - first + 1)
    finally:
        lib.dll.zg_internal_set_slice_bytes(C.c_uint64(0))
        lib.dll.zg_internal_set_encode_chunk_bytes(C.c_uint64(0))
    return count


def _stream_once(lib, d, archive, rng, limit):
    """zg_decompress_stream driven like decode/zstd_iterator.rs:88-153 -> (bytes delivered, input consumed, error code, 0,
    or -1 when the input ran out in the middle of the frame)"""
    from zarc_b200._lib import InBuffer, OutBuffer

    pos, got, calls = 0, b"", 0
    while True:
        n = int(rng.choice([1, 3, 17, 1000, 70_000, 131075]))
        gulp = archive[pos : pos + n]
        if not gulp:
            return got, pos, -1
        ib = C.create_string_buffer(gulp, len(gulp))
        inb = InBuffer(C.cast(ib, C.c_void_p), len(gulp), 0)
        while True:
            cap = int(rng.choice([1, 100, 5000, 131072, 300_000]))
            ob = C.create_string_buffer(cap)
            outb = OutBuffer(C.cast(ob, C.c_void_p), cap, 0)
            r = lib.zg_decompress_stream(d, C.byref(outb), C.byref(inb))
            calls += 1
            assert calls < 200_000, "no progress"
            if lib.zg_is_error(r):
                return got, pos + inb.pos, lib.zg_get_error_code(r)
            got += ob.raw[: outb.pos]
            assert len(got) <= limit, "delivered more than any valid frame of this size could hold"
            if r == 0:
                return got, pos + inb.pos, 0
            if outb.pos < cap and inb.pos == inb.size:
                break
        pos += inb.pos


def streaming(lib, first, count, log=None):
    """Intact and mutated frames (libzstd's and ours) through zg_decompress_stream in random gulps with random output
    capacities, ONE context reused from frame to frame (a frame that failed must leave it usable; only a frame abandoned
    for lack of input gets a new one, as the reference drops its DCtx with the frame iterator).  What the stream delivers
    with a final hint of 0 is exactly what the reference's streaming decoder restores from the same bytes."""
    from tests.test_decode_fuzz_emu import _mutations

    d = lib.zg_dctx_create()
    agree = rejected = 0
    for seed in range(first, first + count):
        rng = np.random.default_rng(seed)
        datas = [text(int(rng.integers(0, 9000)), seed), rand(int(rng.integers(0, 3000)), seed) + bytes(int(rng.integers(0, 5000))),
                 text(int(rng.integers(100_000, 300_000)), seed + 1)]
        for data in datas:
            if rng.integers(0, 2):
                base = ref_path.ref_compress(data, level=int(rng.choice([1, 3, 9])), checksum=bool(rng.integers(0, 2)))
            else:
                base = bytes(compress2(lib, data, level=int(rng.choice([1, 3])), checksum=bool(rng.integers(0, 2))))
            for fr in [base] + _mutations(base, rng, 4):
                archive = fr + b"\x28\xb5\x2f\xfdnext"
                try:
                    ref = ref_path.ref_decompress_stream(archive, 0)
                except ref_path.ZstdError:
                    ref = None
                got, _used, err = _stream_once(lib, d, archive, rng, 128 * 1024 * (len(fr) // 3 + 2))
                if err == 0:
                    assert ref is not None and got == ref, (seed, "accepted what the reference rejects or restores differently")
                    agree += 1
                else:
                    rejected += 1
                    assert fr is not base, (seed, "intact frame refused", err)
                    if err == -1:
                        lib.zg_dctx_free(d)
                        d = lib.zg_dctx_create()
        if log and seed % 10 == 0:
            log(seed, agree + rejected)
    lib.zg_dctx_free(d)
    return agree, rejected


class _DirWriter(ref_container.RefArchiveWriter):
    def directory_bytes(self) -> bytes:
        d = bytearray(ref_container.edition_element())
        for f in self.files:
            if f["digest"] is not None:
                d += ref_container.frame_element(self.enc.frames[f["digest"]])
            d += ref_container.file_element(**f)
        return bytes(d)

    def finalise_with(self, directory: bytes) -> bytes:
        out = bytearray(self.out)
        digest = ref_path._blake3(directory)
        comp = self.enc.compress_frame(directory)
        out += comp
        tb = ref_container.trailer_bytes(digest, -(len(comp) + 8 + 32 + ref_container.EPILOGUE_LENGTH), len(directory))
        out += bytes([0x5F, 0x2A, 0x4D, 0x18]) + struct.pack("<I", len(tb)) + tb
        return bytes(out)


def _mutate_directory(d: bytes, rng) -> bytes:
    f = bytearray(d)
    for _ in range(int(rng.integers(1, 4))):
        kind = int(rng.integers(0, 6))
        n = len(f)
        if n == 0:
            break
        if kind <= 1:
            f[int(rng.integers(0, n))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 2:
            p, m = int(rng.integers(0, n)), int(rng.integers(1, 9))
            f[p : p + m] = bytes(rng.integers(0, 256, m, dtype=np.uint8))
        elif kind == 3:
            f = f[: int(rng.integers(0, n))]
        elif kind == 4:  # a big length / count in front of something
            p = int(rng.integers(0, n))
            f[p : p + 1] = bytes([int(rng.choice([0x5B, 0x9B, 0xBB, 0x7B, 0x1B]))]) + bytes(rng.integers(0, 256, 8, dtype=np.uint8))
        else:  # a run copied somewhere else
            p, q, m = int(rng.integers(0, n)), int(rng.integers(0, n)), int(rng.integers(1, 40))
            f[q:q] = f[p : p + m]
    return bytes(f)


def container_directories(lib_path, first, count, log=None):
    """Archives whose directory element stream was mutated BEFORE it was compressed, digested and given a matching
    trailer (so the reader gets past the integrity checks and has to parse it) through `zarc-b200 list-files` and
    `unpack`: exit code 0 or 1, never a signal, never a hang, nothing written outside the extraction directory."""
    from zarc_b200 import build

    host = build.build_host()
    w = _DirWriter(level=3)
    w.add_file(["a.txt"], text(3000, 1))
    w.add_file(["sub", "b.bin"], rand(2000, 2))
    w.add_file(["sub", "dup.txt"], text(3000, 1))
    w.add_file(["sub", "empty"], b"")
    w.add_file(["big.txt"], text(140_000, 4))
    base = w.directory_bytes()
    env = dict(os.environ, ZARCGPU_LIB=lib_path)
    accepted = 0
    for seed in range(first, first + count):
        rng = np.random.default_rng(seed)
        d = base if seed == first else _mutate_directory(base, rng)
        tmp = tempfile.mkdtemp(prefix="zfuzz")
        try:
            work = os.path.join(tmp, "w")
            os.makedirs(work)
            with open(os.path.join(work, "x.zarc"), "wb") as fh:
                fh.write(w.finalise_with(d))
            for cmd in (["list-files", "x.zarc"], ["unpack", "x.zarc"]):
                p = subprocess.run([host, *cmd], cwd=work, env=env, capture_output=True, timeout=120)  # (a hang raises)
                assert p.returncode in (0, 1), (seed, cmd, p.returncode, p.stderr[-200:])
                if p.returncode == 0 and cmd[0] == "unpack":
                    accepted += 1
            if seed == first:
                assert accepted == 1, "the unmutated archive must unpack"
            assert set(os.listdir(tmp)) == {"w"}, (seed, "something was written outside the extraction directory")
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        if log and seed % 25 == 0:
            log(seed, accepted)
    return accepted


def hostile_metadata(lib, first, count, log=None):
    """zg_unpack_batch_dev / zg_unpack_batch over batches in which some entries carry wild offsets, lengths, sizes or
    output offsets (beyond the archive, beyond the output, 2^63, 2^64 - 1): no crash, every untouched entry still
    decodes (status 0), every wild one is reported in its own status entry.  (On the CPU build "device" pointers are
    host pointers.  The buffers carry 8 bytes of slack: the kernels read aligned 4-byte words, so the word that holds a
    buffer's last byte may be read whole -- never written; see include/zarcgpu.h.)"""
    U = lambda v: np.array([int(x) & (2**64 - 1) for x in v], dtype=object).astype(np.uint64)  # noqa: E731
    for seed in range(first, first + count):
        rng = np.random.default_rng(seed)
        pick = lambda v: int(v[int(rng.integers(0, len(v)))])  # noqa: E731
        datas = [text(int(rng.integers(0, 20000)), seed + i) if rng.integers(0, 2) else rand(int(rng.integers(0, 5000)), seed + i)
                 for i in range(int(rng.integers(1, 12)))]
        frames = [ref_path.ref_compress(d, level=int(rng.choice([1, 3]))) for d in datas]
        archive = bytearray(b"\xaa" * 7)
        off, ln = [], []
        for f in frames:
            off.append(len(archive))
            ln.append(len(f))
            archive += f
        n = len(frames)
        ul = [len(d) for d in datas]
        oo = [int(x) for x in np.cumsum([0] + ul[:-1])]
        total = sum(ul)
        wild = [False] * n
        for k in range(n):
            r = int(rng.integers(0, 8))
            if r == 0:
                off[k] = pick([len(archive) + 5, 2**63, 2**64 - 1, len(archive) - 1])
            elif r == 1:
                ln[k] = pick([0, 1, len(archive) * 2, 2**64 - 1, max(0, ln[k] - 1)])
            elif r == 2:
                ul[k] = pick([ul[k] + 1, max(0, ul[k] - 1) if ul[k] else 5, 2**40, 2**64 - 1])
            elif r == 3:
                oo[k] = pick([total + 1, 2**63, 2**64 - 1])
            wild[k] = r <= 3
        arch = np.frombuffer(bytes(archive) + bytes(8), dtype=np.uint8).copy()
        a_off, a_len, a_ul, a_oo = U(off), U(ln), U(ul), U(oo)
        out = np.zeros(max(total, 1) + 8, dtype=np.uint8)
        ok = np.zeros(n, dtype=np.uint8)
        st = np.zeros(n, dtype=np.uint32)
        dig = np.frombuffer(b"".join(ref_path.c_blake3(d) for d in datas), dtype=np.uint8).copy()
        d = lib.zg_dctx_create()
        rc = lib.zg_unpack_batch_dev(d, arch.ctypes.data, len(archive), n, a_off.ctypes.data, a_len.ctypes.data, a_ul.ctypes.data,
                                     dig.ctypes.data, out.ctypes.data, total, a_oo.ctypes.data, ok.ctypes.data, st.ctypes.data)
        assert (rc == 0) == (not any(wild)) or not any(st), (seed, rc)
        for k in range(n):
            if wild[k]:
                assert st[k] != 0 and ok[k] == 0, (seed, k, "a wild entry went through")
            else:
                assert st[k] == 0 and ok[k] == 1, (seed, k, int(st[k]))
                assert bytes(out[oo[k] : oo[k] + ul[k]]) == datas[k], (seed, k)
        # the host-buffer variant (dense output) on the same metadata: an error code or per-frame statuses, no crash
        lib.zg_unpack_batch(d, arch.ctypes.data, len(archive), n, a_off.ctypes.data, a_len.ctypes.data, a_ul.ctypes.data, dig.ctypes.data,
                            out.ctypes.data, total, None, ok.ctypes.data, st.ctypes.data)
        lib.zg_dctx_free(d)
        if log and seed % 50 == 0:
            log(seed, seed - first + 1)
    return count


def compress_capacity(lib, first, count, log=None):
    """zg_compress2 into destinations of every awkward capacity (0, 1, around the frame header, random, n, the
    reference's n + max(1024, n / 10) of lowlevel_frames.rs:21): either dstSize_tooSmall or a frame of at most `cap`
    bytes that libzstd restores; the destination is an exact-size buffer (an overrun shows under AddressSanitizer)."""
    c = lib.zg_cctx_create()
    lib.check(lib.zg_cctx_init(c, 0))
    made = refused = 0
    for seed in range(first, first + count):
        rng = np.random.default_rng(seed)
        data = glued_input(rng, float(rng.choice([0.05, 0.3, 1.0])))
        n = len(data)
        lib.check(lib.zg_cctx_set_parameter(c, 201, int(rng.integers(0, 2))))
        lib.check(lib.zg_cctx_set_parameter(c, 100, int(rng.choice([1, 3, 9]))))
        bound = n + max(1024, n // 10)
        src = np.frombuffer(data + bytes(8), dtype=np.uint8).copy()
        for cap in sorted({0, 1, 12, 13, 14, int(rng.integers(0, bound + 1)), int(rng.integers(0, bound + 1)), n // 3, n, n + 3, n + 16, bound}):
            dst = np.full(max(cap, 1), 0xEE, dtype=np.uint8)
            r = lib.zg_compress2(c, dst.ctypes.data, cap, src.ctypes.data, n)
            if lib.zg_is_error(r):
                assert lib.zg_get_error_code(r) == 70, (seed, cap, lib.zg_get_error_code(r))
                refused += 1
            else:
                assert r <= cap and ref_path.ref_decompress(bytes(dst[:r]), n) == data, (seed, cap)
                made += 1
        full = np.zeros(bound, dtype=np.uint8)
        assert not lib.zg_is_error(lib.zg_compress2(c, full.ctypes.data, bound, src.ctypes.data, n)), (seed, "the reference's capacity must do")
        if log and seed % 20 == 0:
            log(seed, made + refused)
    lib.zg_cctx_free(c)
    return made, refused

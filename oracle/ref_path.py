"""ORACLE — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The reference's content path, restated call-for-call on the *same third-party libraries at the
same versions* the reference links (they are not vendored under /root/reference):

* libzstd 1.5.5  (zstd-sys 2.0.9+zstd.1.5.5, Cargo.lock:2480-2481)  -> /lib/x86_64-linux-gnu/libzstd.so.1
* BLAKE3         (crate blake3 1.5.0, Cargo.lock:191-192)           -> Python package `blake3` (same Rust core)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import
this module.  It is also what generated tests/golden/*.json (tests/golden/make_golden.py).

`RefEncoder` follows crates/zarc/src/encode.rs:58-97 + encode/content_frame.rs:20-60 +
encode/lowlevel_frames.rs:19-39; `RefDecoder.read_content_frame` follows
crates/zarc/src/decode/zstd_iterator.rs:88-153 + decode/frame_iterator.rs:94-103,77-88.
"""
from __future__ import annotations

import ctypes
import ctypes.util
import os
import subprocess
from dataclasses import dataclass

_HERE = os.path.dirname(os.path.abspath(__file__))

# --------------------------------------------------------------------------------------------
# libzstd 1.5.5
_zstd = ctypes.CDLL("libzstd.so.1")
_zstd.ZSTD_versionNumber.restype = ctypes.c_uint
ZSTD_VERSION = _zstd.ZSTD_versionNumber()

_sz = ctypes.c_size_t
_vp = ctypes.c_void_p
for _n, _res, _args in [
    ("ZSTD_createCCtx", _vp, []),
    ("ZSTD_freeCCtx", _sz, [_vp]),
    ("ZSTD_initCStream", _sz, [_vp, ctypes.c_int]),
    ("ZSTD_CCtx_setParameter", _sz, [_vp, ctypes.c_int, ctypes.c_int]),
    ("ZSTD_CCtx_reset", _sz, [_vp, ctypes.c_int]),
    ("ZSTD_compress2", _sz, [_vp, _vp, _sz, _vp, _sz]),
    ("ZSTD_createDCtx", _vp, []),
    ("ZSTD_freeDCtx", _sz, [_vp]),
    ("ZSTD_decompressStream", _sz, [_vp, _vp, _vp]),
    ("ZSTD_decompressDCtx", _sz, [_vp, _vp, _sz, _vp, _sz]),
    ("ZSTD_isError", ctypes.c_uint, [_sz]),
    ("ZSTD_getErrorName", ctypes.c_char_p, [_sz]),
    ("ZSTD_DStreamInSize", _sz, []),
    ("ZSTD_DStreamOutSize", _sz, []),
    ("ZSTD_findFrameCompressedSize", _sz, [_vp, _sz]),
    ("ZSTD_getFrameContentSize", ctypes.c_ulonglong, [_vp, _sz]),
]:
    _f = getattr(_zstd, _n)
    _f.restype = _res
    _f.argtypes = _args

# libzstd enum values (zstd.h 1.5.5)
ZSTD_c_compressionLevel = 100
ZSTD_c_windowLog = 101
ZSTD_c_contentSizeFlag = 200
ZSTD_c_checksumFlag = 201
ZSTD_reset_session_only = 1


class ZstdError(RuntimeError):
    pass


def _check(code: int) -> int:
    if _zstd.ZSTD_isError(code):
        raise ZstdError(_zstd.ZSTD_getErrorName(code).decode())
    return code


class _Buf(ctypes.Structure):  # ZSTD_inBuffer / ZSTD_outBuffer share this layout
    _fields_ = [("ptr", _vp), ("size", _sz), ("pos", _sz)]


def _blake3(data) -> bytes:
    import blake3

    return blake3.blake3(data, max_threads=1).digest()


@dataclass
class RefFrame:  # crates/zarc/src/directory/frame.rs:12-32
    edition: int
    offset: int
    digest: bytes
    length: int
    uncompressed: int


class RefEncoder:
    """`Encoder` restated (content path only).  `out` is a bytearray playing the writer."""

    FILE_MAGIC = bytes([0x50, 0x2A, 0x4D, 0x18, 0x04, 0x00, 0x00, 0x00, 0x65, 0xAA, 0xDC, 0x01])  # header.rs:35-40

    def __init__(self, out: bytearray, *, checksum: bool = True, level: int | None = None):
        self.out = out
        self.cctx = _zstd.ZSTD_createCCtx()  # encode.rs:61
        _check(_zstd.ZSTD_initCStream(self.cctx, 0))  # encode.rs:62  (CCtx::init(0))
        out += self.FILE_MAGIC  # encode.rs:65
        self.offset = len(self.FILE_MAGIC)
        self.frames: dict[bytes, RefFrame] = {}
        self.order: list[bytes] = []
        if checksum:  # crates/zarc-cli/src/pack.rs:227
            self.set_zstd_parameter(ZSTD_c_checksumFlag, 1)
        if level is not None:  # pack.rs:229-232
            self.set_zstd_parameter(ZSTD_c_compressionLevel, level)

    def __del__(self):
        if getattr(self, "cctx", None):
            _zstd.ZSTD_freeCCtx(self.cctx)
            self.cctx = None

    def set_zstd_parameter(self, param: int, value: int) -> None:  # encode.rs:84-89
        _check(_zstd.ZSTD_CCtx_setParameter(self.cctx, param, value))

    def compress_frame(self, content: bytes) -> bytes:  # lowlevel_frames.rs:19-39
        n = len(content)
        cap = n + max(1024, n // 10)
        if cap > getattr(self, "_dst_cap", 0):  # one reusable destination (the Rust side allocates a Vec per frame)
            self._dst = ctypes.create_string_buffer(cap)
            self._dst_cap = cap
        r = _check(_zstd.ZSTD_compress2(self.cctx, self._dst, cap, bytes(content) if n else None, n))
        return ctypes.string_at(self._dst, r)

    def add_data_frame(self, content: bytes) -> bytes:  # content_frame.rs:20-60
        offset = self.offset
        digest = _blake3(content)  # :26
        if digest in self.frames:  # :30
            return digest
        _check(_zstd.ZSTD_CCtx_reset(self.cctx, ZSTD_reset_session_only))  # :37-39
        frame = self.compress_frame(content)  # :41
        self.out += frame
        self.offset += len(frame)  # :45
        self.frames[digest] = RefFrame(1, offset, digest, len(frame), len(content))  # :48-57
        self.order.append(digest)
        return digest


def ref_compress(content: bytes, level: int = 3, checksum: bool = True) -> bytes:
    """One frame exactly as the reference's Encoder would write it."""
    out = bytearray()
    enc = RefEncoder(out, checksum=checksum, level=level)
    _check(_zstd.ZSTD_CCtx_reset(enc.cctx, ZSTD_reset_session_only))
    return enc.compress_frame(content)


def ref_decompress_stream(archive: bytes, offset: int) -> bytes:
    """zstd_iterator.rs:88-153: new DCtx, <=131075-byte gulps, >=131072-byte output chunks."""
    dctx = _zstd.ZSTD_createDCtx()
    try:
        in_size = max(_zstd.ZSTD_DStreamInSize(), 1024)
        out_size = max(_zstd.ZSTD_DStreamOutSize(), 1024)
        pos = offset
        chunks = []
        done = False
        base = ctypes.cast(ctypes.c_char_p(archive), _vp).value if isinstance(archive, bytes) else None
        outmem = ctypes.create_string_buffer(out_size)
        out_addr = ctypes.cast(outmem, _vp)
        while not done:
            avail = min(in_size, len(archive) - pos)
            if avail <= 0:
                raise ZstdError("unexpected end of archive")
            if base is not None:  # read straight from the archive bytes (the reference reads into a fresh 131 075-byte Vec)
                inbuf = _Buf(base + pos, avail, 0)
            else:
                inbuf_mem = ctypes.create_string_buffer(bytes(archive[pos : pos + avail]), avail)
                inbuf = _Buf(ctypes.cast(inbuf_mem, _vp), avail, 0)
            while True:
                outbuf = _Buf(out_addr, out_size, 0)
                hint = _check(_zstd.ZSTD_decompressStream(dctx, ctypes.byref(outbuf), ctypes.byref(inbuf)))
                chunks.append(ctypes.string_at(out_addr, outbuf.pos))
                if hint == 0:
                    done = True
                    break
                if outbuf.pos < out_size and inbuf.pos == inbuf.size:
                    break
            pos += inbuf.pos
        return b"".join(chunks)
    finally:
        _zstd.ZSTD_freeDCtx(dctx)


def ref_stream_digest(archive, offset: int = 0):
    """FrameIterator drained without keeping the bytes (decode/frame_iterator.rs:94-103: every chunk the streaming
    decoder hands out goes into the Hasher; :77 finalize): returns (BLAKE3 digest, bytes produced, bytes consumed).
    `archive` may be bytes or a numpy u8 array (multi-GiB frames)."""
    import blake3
    import numpy as np

    if isinstance(archive, (bytes, bytearray)):
        archive = np.frombuffer(archive, dtype=np.uint8)
    base = archive.ctypes.data
    total = int(archive.shape[0])
    dctx = _zstd.ZSTD_createDCtx()
    try:
        in_size = max(_zstd.ZSTD_DStreamInSize(), 1024)
        out_size = max(_zstd.ZSTD_DStreamOutSize(), 1024)
        outmem = ctypes.create_string_buffer(out_size)
        out_addr = ctypes.cast(outmem, _vp)
        hasher = blake3.blake3(max_threads=1)
        pos, produced, done = offset, 0, False
        while not done:
            avail = min(in_size, total - pos)
            if avail <= 0:
                raise ZstdError("unexpected end of archive")
            inbuf = _Buf(base + pos, avail, 0)
            while True:
                outbuf = _Buf(out_addr, out_size, 0)
                hint = _check(_zstd.ZSTD_decompressStream(dctx, ctypes.byref(outbuf), ctypes.byref(inbuf)))
                if outbuf.pos:
                    hasher.update(ctypes.string_at(out_addr, outbuf.pos))
                    produced += outbuf.pos
                if hint == 0:
                    done = True
                    break
                if outbuf.pos < out_size and inbuf.pos == inbuf.size:
                    break
            pos += inbuf.pos
        return hasher.digest(), produced, pos - offset
    finally:
        _zstd.ZSTD_freeDCtx(dctx)


def ref_decompress(frame: bytes, max_out: int) -> bytes:
    """One-shot libzstd decode (the "reference zstd decoder" for GPU-made frames)."""
    dctx = _zstd.ZSTD_createDCtx()
    try:
        dst = ctypes.create_string_buffer(max(max_out, 1))
        src = ctypes.create_string_buffer(bytes(frame), len(frame))
        r = _check(_zstd.ZSTD_decompressDCtx(dctx, dst, max_out, src, len(frame)))
        return dst.raw[:r]
    finally:
        _zstd.ZSTD_freeDCtx(dctx)


def find_frame_compressed_size(buf: bytes) -> int:
    src = ctypes.create_string_buffer(bytes(buf), len(buf))
    return _check(_zstd.ZSTD_findFrameCompressedSize(src, len(buf)))


class RefDecoder:
    """`Decoder::read_content_frame` + `FrameIterator` restated."""

    def __init__(self, archive: bytes, frames: dict[bytes, RefFrame]):
        self.archive = archive
        self.frames = frames

    def read_content_frame(self, digest: bytes):  # frame_iterator.rs:14-27
        entry = self.frames.get(digest)
        if entry is None:
            return None
        data = ref_decompress_stream(self.archive, entry.offset)
        ok = _blake3(data) == digest  # frame_iterator.rs:77,86-88
        return data, ok


# --------------------------------------------------------------------------------------------
# the plain-C restatement (oracle/zarc_oracle.c)
def build_c_oracle(force: bool = False) -> str:
    so = os.path.join(_HERE, "libzarc_oracle.so")
    src = os.path.join(_HERE, "zarc_oracle.c")
    if force or not os.path.exists(so) or (os.path.exists(src) and os.path.getmtime(so) < os.path.getmtime(src)):
        tmp = f"{so}.{os.getpid()}.tmp"  # (atomic: several processes may load or rebuild it at once)
        try:
            subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-o", tmp, src])
            os.replace(tmp, so)
        finally:
            if os.path.exists(tmp):
                os.unlink(tmp)
    return so


LIT_TYPES = ("raw", "rle", "huf", "treeless")  # Literals_Block_Type 0..3
SEQ_TABLES = ("ll", "of", "ml")                # in the order of the Symbol_Compression_Modes byte
SEQ_MODES = ("predefined", "rle", "fse", "repeat")
NONE_SEEN = (1 << 64) - 1                      # regen_min_*, min_match and huf_min_nw while there was none


def lit_header_bytes(st: dict, kind: str) -> dict:
    """Literals sections of `kind` ("raw", "rle", "huf" or "treeless") per header size in bytes.  Raw / RLE: Size_Format
    0 and 2 are 1 byte, 1 is 2 bytes, 3 is 3 bytes.  Compressed: Size_Format 0 (1 stream) and 1 (4 streams) are 3 bytes,
    2 is 4 and 3 is 5."""
    f = [st[f"lit_{kind}_sf{k}"] for k in range(4)]
    if kind in ("raw", "rle"):
        return {1: f[0] + f[2], 2: f[1], 3: f[3]}
    return {3: f[0] + f[1], 4: f[2], 5: f[3]}


class _Stats(ctypes.Structure):
    _fields_ = [
        (n, ctypes.c_uint64)
        for n in (
            "blocks_raw blocks_rle blocks_compressed lit_raw lit_rle lit_huf1 lit_huf4 lit_treeless "
            "seq_predefined seq_rle seq_fse seq_repeat sequences rep_offsets window_size has_checksum single_segment "
            + " ".join(f"lit_{t}_sf{f}" for t in LIT_TYPES for f in range(4))
            + " huf_max_bits huf_wdirect huf_wfse "
            + " ".join(f"regen_max_{t}" for t in LIT_TYPES) + " "
            + " ".join(f"regen_min_{t}" for t in LIT_TYPES)
            + " nseq_h1 nseq_h2 nseq_h3 max_ll_code max_ml_code max_of_code "
            + " ".join(f"{t}_{m}" for t in SEQ_TABLES for m in SEQ_MODES)
            + " max_ll_log max_of_log max_ml_log min_match max_match max_offset max_lit_run xblock_matches xblock_reps "
            "fcs_size blocks huf_max_sym huf_min_nw huf_max_nsym"
        ).split()
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


_c = None


def c_oracle():
    global _c
    if _c is None:
        _c = ctypes.CDLL(build_c_oracle())
        _c.zo_blake3.argtypes = [_vp, _sz, _vp]
        _c.zo_blake3.restype = None
        _c.zo_xxh64.argtypes = [_vp, _sz, ctypes.c_uint64]
        _c.zo_xxh64.restype = ctypes.c_uint64
        _c.zo_zstd_decompress_frame.argtypes = [_vp, _sz, _vp, _sz, ctypes.POINTER(_sz), ctypes.POINTER(_Stats)]
        _c.zo_zstd_decompress_frame.restype = _sz
        _c.zo_is_error.argtypes = [_sz]
    return _c


def c_blake3(data: bytes) -> bytes:
    out = ctypes.create_string_buffer(32)
    c_oracle().zo_blake3(ctypes.c_char_p(bytes(data)), len(data), out)
    return out.raw


def c_xxh64(data: bytes, seed: int = 0) -> int:
    return c_oracle().zo_xxh64(ctypes.c_char_p(bytes(data)), len(data), seed)


def c_zstd_decompress_frame(frame: bytes, cap: int):
    """Returns (data | None, error_code, consumed, stats)."""
    dst = ctypes.create_string_buffer(max(cap, 1))
    consumed = _sz(0)
    st = _Stats()
    r = c_oracle().zo_zstd_decompress_frame(ctypes.c_char_p(bytes(frame)), len(frame), dst, cap, ctypes.byref(consumed), ctypes.byref(st))
    if c_oracle().zo_is_error(r):
        return None, (1 << 64) - r, 0, st.as_dict()
    return dst.raw[:r], 0, consumed.value, st.as_dict()

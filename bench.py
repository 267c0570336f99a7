#!/usr/bin/env python
"""bench.py -- pack & unpack GB/s (uncompressed) of the zarc content path on B200.

A "step" = one pass of the hot path over one batch: pack the rank's shard of the synthetic corpus
(BLAKE3 digests -> dedup -> Zstandard frame encode -> offsets -> frames) and then unpack it again
(Zstandard frame decode -> checksum -> BLAKE3 verify), device-resident.  `value` = uncompressed
corpus bytes through that pack+unpack round trip per second, summed over ranks (so a corpus of B
bytes per rank that packs in tp and unpacks in tu gives N*B/(tp+tu)); `pack_gbs` / `unpack_gbs`
are the two legs on their own.  `e2e` is the same round trip through the host-buffer C ABI
(zg_pack_batch / zg_unpack_batch) with pinned host buffers and every H2D/D2H copy inside the timed
region.  `--impl reference` times the reference's own CPU path (oracle/ref_path.py: libzstd 1.5.5 +
BLAKE3 with the reference's call sequence) on the host cores.

Workloads (BASELINE.json configs; SURVEY.md 8d): `--config c2` (default, the headline: ~1M files of
1-64 KiB, 10.2 GB per GPU), `c1` (2 000 files, 256 MiB), `c3` (8 x 4 GiB logs), `c4` (20 GB, 50 %
duplicate files), `c5` (unpack + verify of frames made by the REFERENCE path at levels 1/3/9 over a
C2+C1+C3-shaped mix, replicated on the device to 50 GB).  The default run also measures, as `extras`
of the same JSON line, C2 strong-scaled (one 10.2 GB corpus over all ranks, N > 1), C4, C3 and C5.

Multi-GPU (one rank per GPU, NCCL): files are sharded by `zarc_b200.parallel.ShardPlan`; the timed
pack step holds the whole exchange -- BLAKE3, all-gather of digests, global first-occurrence
decisions, encode, all-gather of frame sizes, archive offsets.  No content bytes cross GPUs.

Launch: `python bench.py --gpus 1` or under torchrun for N > 1.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pack+unpack round-trip GB/s (uncompressed)"


# ------------------------------------------------------------------------------------------------
# CPU reference arm (also the cpu_baseline of the GPU arm).  Runs BEFORE any CUDA initialisation and
# never loads the product library: the corpus comes from tools/libzarc_corpus.so (the generator alone).
def _cpu_files(kind: str, seed: int, total_bytes: int, wid: int, nworkers: int):
    from zarc_b200 import corpus

    c = corpus.c5_mix(total_bytes=total_bytes, seed=seed) if kind == "c5" else corpus.c2_source_tree(total_bytes=total_bytes, seed=seed)
    # dealt largest first so that the few big files of the C5 mix spread over the workers
    order = np.argsort(-c.len.astype(np.int64), kind="stable")
    idx = np.sort(order[wid::nworkers])
    sub = corpus.take(c, idx)
    blob = corpus.materialise_standalone(sub)
    return idx, sub, [bytes(blob[int(o) : int(o) + int(l)]) for o, l in zip(sub.off, sub.len)]


def _cpu_worker(args):
    """One host core: generate its share of the sample, then time the reference path on it."""
    seed, total_bytes, level, wid, nworkers = args
    from oracle import ref_path

    _, sub, files = _cpu_files("c2", seed, total_bytes, wid, nworkers)
    out = bytearray()
    t0 = time.perf_counter()
    enc = ref_path.RefEncoder(out, checksum=True, level=level)
    digests = [enc.add_data_frame(f) for f in files]
    t1 = time.perf_counter()
    dec = ref_path.RefDecoder(bytes(out), enc.frames)
    ok = True
    for d, f in zip(digests, files):
        data, good = dec.read_content_frame(d)
        ok = ok and good and len(data) == len(f)
    t2 = time.perf_counter()
    return sub.total_bytes, len(out) - 12, t1 - t0, t2 - t1, ok


def cpu_reference_run(seed: int, sample_bytes: int, level: int, cores: int):
    """All host cores, one process each over disjoint files of the sample (the reference itself is
    single-threaded; this is the generous aggregate).  Returns dict(value GB/s round trip, ...)."""
    import multiprocessing as mp

    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(seed, sample_bytes, level, w, cores) for w in range(cores)])
    nbytes = sum(r[0] for r in res)
    cbytes = sum(r[1] for r in res)
    tp = max(r[2] for r in res)
    tu = max(r[3] for r in res)
    assert all(r[4] for r in res), "reference round trip failed"
    return dict(bytes=nbytes, ratio=nbytes / max(cbytes, 1), pack_gbs=nbytes / tp / 1e9, unpack_gbs=nbytes / tu / 1e9,
                value=nbytes / (tp + tu) / 1e9, pack_s=tp, unpack_s=tu)


def _ratio_worker(args):
    seed, total_bytes, levels, wid, nworkers = args
    from oracle import ref_path

    _, sub, files = _cpu_files("c2", seed, total_bytes, wid, nworkers)
    return sub.total_bytes, {lv: sum(len(ref_path.ref_compress(f, level=lv)) for f in files) for lv in levels}


def cpu_ratio_run(seed: int, sample_bytes: int, levels, cores: int):
    """libzstd's ratio at each level on a C2 sample (the reference's call sequence), for the line's `levels` table."""
    import multiprocessing as mp

    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        res = pool.map(_ratio_worker, [(seed, sample_bytes, tuple(levels), w, cores) for w in range(cores)])
    n = sum(r[0] for r in res)
    return {lv: n / max(1, sum(r[1][lv] for r in res)) for lv in levels}


def _c5_worker(args):
    """One host core of the C5 producer: frames made the reference's way (RefEncoder call sequence) at each level over
    this worker's files of the mix, and the reference's own unpack + verify of them, timed."""
    seed, total_bytes, levels, wid, nworkers = args
    from oracle import ref_path

    idx, sub, files = _cpu_files("c5", seed, total_bytes, wid, nworkers)
    out = {}
    for level in levels:
        t0 = time.perf_counter()
        frames = [ref_path.ref_compress(f, level=level) for f in files]
        t1 = time.perf_counter()
        arch = b"".join(frames)
        pos, ok = 0, True
        for f, fr in zip(files, frames):
            data = ref_path.ref_decompress_stream(arch, pos)  # zstd_iterator.rs:88-153 call sequence
            ok = ok and ref_path._blake3(data) == ref_path._blake3(f)  # frame_iterator.rs:77,86-88
            pos += len(fr)
        t2 = time.perf_counter()
        out[level] = (arch, np.array([len(fr) for fr in frames], dtype=np.uint64), t1 - t0, t2 - t1, ok)
    digests = b"".join(ref_path._blake3(f) for f in files)
    return idx, sub.len.copy(), digests, out


def c5_produce(seed: int, total_bytes: int, levels, cores: int):
    """-> dict(level -> dict(archive u8[], off, len, ulen, digests, global file idx, cpu pack / unpack seconds))."""
    import multiprocessing as mp

    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        res = pool.map(_c5_worker, [(seed, total_bytes, tuple(levels), w, cores) for w in range(cores)])
    out = {}
    idx = np.concatenate([r[0] for r in res])
    ulen = np.concatenate([r[1] for r in res])
    dig = np.frombuffer(b"".join(r[2] for r in res), dtype=np.uint8)
    for level in levels:
        arch = np.frombuffer(b"".join(r[3][level][0] for r in res), dtype=np.uint8)
        flen = np.concatenate([r[3][level][1] for r in res])
        assert all(r[3][level][4] for r in res), "reference unpack of its own frames failed"
        out[level] = dict(archive=arch, len=flen, off=(np.cumsum(flen) - flen).astype(np.uint64), ulen=ulen, digests=dig, idx=idx,
                          cpu_pack_s=max(r[3][level][2] for r in res), cpu_unpack_s=max(r[3][level][3] for r in res))
    return out


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(s[1])) for s in self.samples if len(s) > 8 and s[1].replace(".", "").isdigit())
        mx = [int(float(s[2])) for s in self.samples if len(s) > 8 and s[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            if len(s) > 8:
                for name, v in zip(names, s[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=sorted(reasons),
                    samples=len(self.samples))


def measured_peaks():
    """(hbm GB/s, source, int32 lane-ops/s or None): the driver-written HBM peak and this repo's INT32-issue peak."""
    hbm, src = 6650.0, "fallback (B200_PROFILING.md)"
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            hbm, src = float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return hbm, src


def ncu_traffic(kernel: str, input_bytes_per_launch: float | None = None):
    """DRAM bytes per launch from the committed `ncu --set full` capture of this kernel, or None.  The capture names the
    input bytes of ITS launch (`corpus_bytes`); a launch of this run that covers a different amount of input (the encoder
    works in chunks) is charged in proportion."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        try:
            e = json.load(open(p)).get(kernel, {})
            t = e.get("dram_bytes_per_launch")
            if t and input_bytes_per_launch and e.get("corpus_bytes"):
                t = t * input_bytes_per_launch / e["corpus_bytes"]
            return t
        except Exception:
            return None
    return None


def workload_text(config: str, args, world: int, scaling: str) -> str:
    if config == "c2":
        per = f"{args.corpus_gb:g} GB uncompressed per GPU" if scaling == "weak" else f"{args.corpus_gb:g} GB uncompressed in total, sharded over {world} GPU(s)"
        return (f"C2 synthetic source-tree corpus: {per} (~{int(args.corpus_gb * 1e9 / 10240):,} files of 1-64 KiB per {args.corpus_gb:g} GB, "
                f"80% src / 15% text / 5% random), zstd level {args.level}, checksumFlag=1")
    if config == "c1":
        return f"C1 synthetic tree: 2,000 files of 4 KiB-1 MiB (256 MiB, even text / odd random), zstd level {args.level}, checksumFlag=1"
    if config == "c3":
        return (f"C3: {args.c3_files} x {args.c3_file_gib:g} GiB semi-compressible log files, one frame per file, sharded over {world} GPU(s), "
                f"zstd level {args.level}, checksumFlag=1")
    if config == "c4":
        return (f"C4 dedup-heavy corpus: {args.c4_gb:g} GB, C2-shaped, every odd file a byte copy of the preceding even file (50 % duplicates), "
                f"sharded over {world} GPU(s), zstd level {args.level}, checksumFlag=1")
    return (f"C5: unpack + verify of frames made by the reference path (libzstd 1.5.5, RefEncoder call sequence) at levels 1/3/9 over a "
            f"C2+C1+C3-shaped mix of {args.c5_unique_gb:g} GB unique per level, replicated on the device to {args.c5_total_gb:g} GB in total")


# ------------------------------------------------------------------------------------------------
class Ctx:
    """What every leg needs: the library, the device, the process group."""

    def __init__(self, lib, torch, dist, rank, world, local_rank):
        self.lib, self.torch, self.dist = lib, torch, dist
        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.dev = torch.device("cuda", local_rank)
        self.stream = torch.cuda.current_stream().cuda_stream

    def to_dev(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def rank_max(self, v):
        if self.world == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def rank_sum(self, v):
        if self.world == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def ev(self):
        return self.torch.cuda.Event(enable_timing=True)


class RoundTrip:
    """Device-resident pack + unpack of this rank's shard of a corpus."""

    def __init__(self, cx: Ctx, glob, level: int, checksum: bool = True, partition: str = "auto"):
        from zarc_b200 import corpus, parallel

        torch, lib = cx.torch, cx.lib
        self.cx, self.parallel = cx, parallel
        self.plan = parallel.ShardPlan(glob.len, cx.world, mode=partition)
        self.mine = corpus.take(glob, self.plan.mine(cx.rank), name=f"{glob.name}[rank {cx.rank}]")
        m = self.mine
        self.n, self.B = m.n_files, m.total_bytes
        so, sl, sk, key = m.segments()
        self.blob = torch.empty(m.blob_bytes + 64, dtype=torch.uint8, device=cx.dev)
        segs = [cx.to_dev(x) for x in (so, sl, sk, key)]
        lib.check(lib.zg_corpus_generate_dev(cx.stream, self.blob.data_ptr(), segs[0].data_ptr(), segs[1].data_ptr(), segs[2].data_ptr(),
                                             segs[3].data_ptr(), len(so)))
        torch.cuda.synchronize()
        del segs
        self.off, self.ln = cx.to_dev(m.off.astype(np.int64)), cx.to_dev(m.len.astype(np.int64))
        self.cctx, self.dctx = lib.zg_cctx_create(), lib.zg_dctx_create()
        assert self.cctx and self.dctx
        lib.check(lib.zg_cctx_set_stream(self.cctx, cx.stream))
        lib.check(lib.zg_dctx_set_stream(self.dctx, cx.stream))
        lib.check(lib.zg_cctx_init(self.cctx, 0))  # encode.rs:62
        lib.check(lib.zg_cctx_set_parameter(self.cctx, 201, 1 if checksum else 0))  # ChecksumFlag, pack.rs:227 / :92
        lib.check(lib.zg_cctx_set_parameter(self.cctx, 100, level))  # pack.rs:229-232
        n, B = self.n, self.B
        self.cap = B + max(1024, B // 10) + 32 * n + 4096
        i64, u8 = torch.int64, torch.uint8
        self.d_dig = torch.empty(max(n, 1) * 32, dtype=u8, device=cx.dev)
        self.d_first = torch.empty(max(n, 1), dtype=u8, device=cx.dev)
        self.d_foff = torch.empty(max(n, 1), dtype=i64, device=cx.dev)
        self.d_flen = torch.empty(max(n, 1), dtype=i64, device=cx.dev)
        self.d_frames = torch.empty(self.cap, dtype=u8, device=cx.dev)
        self.d_out = torch.empty(m.blob_bytes + 64, dtype=u8, device=cx.dev)
        self.d_ok = torch.zeros(max(n, 1), dtype=u8, device=cx.dev)
        self.d_status = torch.zeros(max(n, 1), dtype=torch.int32, device=cx.dev)
        self.nbytes = np.zeros(1, dtype=np.uint64)
        self.total = None      # archive end offset (device scalar) after the last pack
        self.sel = None        # unpack list (multi-GPU with duplicates held by other ranks)
        self.host_ms = []      # N > 1: per pack, host wall clock of [digests, dedup exchange, encode, offsets exchange]

    def pack(self):
        cx, lib = self.cx, self.cx.lib
        if cx.world == 1:
            lib.check(lib.zg_cctx_reset_archive(self.cctx, 12))
            lib.check(lib.zg_pack_batch_dev(self.cctx, self.blob.data_ptr(), self.off.data_ptr(), self.ln.data_ptr(), self.n, self.d_dig.data_ptr(),
                                            self.d_first.data_ptr(), self.d_foff.data_ptr(), self.d_flen.data_ptr(), self.d_frames.data_ptr(),
                                            self.cap, self.nbytes.ctypes.data))
            return
        # (1) digests (content_frame.rs:26) -> (2) all-gather + first-occurrence decisions over the GLOBAL order (:30)
        t0 = time.perf_counter()
        lib.check(lib.zg_blake3_batch_dev(cx.stream, self.blob.data_ptr(), self.off.data_ptr(), self.ln.data_ptr(), self.n, self.d_dig.data_ptr()))
        t1 = time.perf_counter()
        first_l, _, first_g, rep_g = self.parallel.global_dedup(lib, self.plan, self.d_dig[: self.n * 32].view(self.n, 32), stream=cx.stream)
        t2 = time.perf_counter()
        # (3) encode what this rank is first for (:41) -> (4) all-gather of frame sizes, offsets in insertion order (:22,45)
        lib.check(lib.zg_cctx_reset_archive(self.cctx, 0))
        sel = first_l.contiguous()
        lib.check(lib.zg_pack_batch_dev_ex(self.cctx, self.blob.data_ptr(), self.off.data_ptr(), self.ln.data_ptr(), self.n, self.d_dig.data_ptr(),
                                           sel.data_ptr(), None, self.d_first.data_ptr(), self.d_foff.data_ptr(), self.d_flen.data_ptr(),
                                           self.d_frames.data_ptr(), self.cap, self.nbytes.ctypes.data))
        t3 = time.perf_counter()
        flen_local = self.d_flen[: self.n] * self.d_first[: self.n].to(cx.torch.int64)
        self.g_off, self.g_len, self.total = self.parallel.global_offsets(lib, self.plan, flen_local, first_g, rep_g, base=12, stream=cx.stream)
        # host-side wall clock of the four parts of a multi-GPU pack (the library calls block until their results are on the host)
        self.host_ms.append([round((b - a) * 1e3, 2) for a, b in ((t0, t1), (t1, t2), (t2, t3), (t3, time.perf_counter()))])

    def prepare_unpack(self):
        """After a pack: which files this rank restores (all of them, except duplicates whose only frame another rank holds)."""
        torch = self.cx.torch
        base = 12 if self.cx.world == 1 else 0
        have = self.d_flen[: self.n] > 0
        if bool(have.all()):
            self.u_n, self.u_off, self.u_len = self.n, (self.d_foff[: self.n] - base).contiguous(), self.d_flen
            self.u_ulen, self.u_dig, self.u_oo, self.u_bytes = self.ln, self.d_dig, self.off, self.B
        else:
            k = torch.nonzero(have).flatten()
            self.u_n = int(k.numel())
            self.u_off, self.u_len = (self.d_foff[k] - base).contiguous(), self.d_flen[k].contiguous()
            self.u_ulen, self.u_oo = self.ln[k].contiguous(), self.off[k].contiguous()
            self.u_dig = self.d_dig[: self.n * 32].view(self.n, 32)[k].contiguous()
            self.u_bytes = int(self.u_ulen.sum().item())
            self.u_keep = k

    def unpack(self):
        lib = self.cx.lib
        lib.check(lib.zg_unpack_batch_dev(self.dctx, self.d_frames.data_ptr(), int(self.nbytes[0]), self.u_n, self.u_off.data_ptr(), self.u_len.data_ptr(),
                                          self.u_ulen.data_ptr(), self.u_dig.data_ptr(), self.d_out.data_ptr(), self.mine.blob_bytes,
                                          self.u_oo.data_ptr(), self.d_ok.data_ptr(), self.d_status.data_ptr()))

    def verify(self):
        torch = self.cx.torch
        assert int(self.d_ok[: self.u_n].sum().item()) == self.u_n and int(self.d_status[: self.u_n].abs().sum().item()) == 0, "unpack verification failed"
        if self.u_n == self.n:
            nb, step = self.mine.blob_bytes, 1 << 30  # (in pieces: torch.equal materialises a temporary as large as its inputs)
            for o in range(0, nb, step):
                assert torch.equal(self.d_out[o : min(nb, o + step)], self.blob[o : min(nb, o + step)]), "round trip is not byte-identical"

    def free(self):
        self.cx.lib.zg_cctx_free(self.cctx)
        self.cx.lib.zg_dctx_free(self.dctx)
        for k in list(self.__dict__):
            if k.startswith(("d_", "u_", "g_")) or k in ("blob", "off", "ln", "sel"):
                self.__dict__[k] = None
        self.cx.torch.cuda.empty_cache()


def time_roundtrip(cx: Ctx, rt: RoundTrip, steps: int, warmup: int):
    """-> (ms per step, pack ms, unpack ms), each the max over ranks of the device time (CUDA events)."""
    for i in range(warmup):
        rt.pack()
        if i == 0:
            rt.prepare_unpack()
        rt.unpack()
    if warmup == 0:
        rt.pack()
        rt.prepare_unpack()
    cx.sync_all()
    rt.verify()
    e0, e1 = cx.ev(), cx.ev()
    pk, up = [], []
    cx.sync_all()
    e0.record()
    for _ in range(steps):
        a, b, c = cx.ev(), cx.ev(), cx.ev()
        a.record()
        rt.pack()
        b.record()
        rt.unpack()
        c.record()
        pk.append((a, b))
        up.append((b, c))
    e1.record()
    cx.sync_all()
    total = cx.rank_max(e0.elapsed_time(e1)) / steps
    tp = cx.rank_max(sum(x.elapsed_time(y) for x, y in pk) / steps)
    tu = cx.rank_max(sum(x.elapsed_time(y) for x, y in up) / steps)
    rt.step_ms = {"pack": [round(x.elapsed_time(y), 2) for x, y in pk], "unpack": [round(x.elapsed_time(y), 2) for x, y in up]}
    if rt.host_ms:
        rt.step_ms["pack_host_parts[digests,dedup_exchange,encode,offsets_exchange]"] = rt.host_ms[-steps:]
    return total, tp, tu


def dump_outputs(rt: RoundTrip, out_dir: str, max_files: int = 1 << 16, max_bytes: int = 1 << 22, seed: int = 7):
    """Write what the last pack + unpack handed its caller to out_dir/<name>.npy (float32, or float64 where values pass
    2^24), so that two builds run with the same arguments can be compared array for array.  Per-file arrays keep a seeded
    sample of at most `max_files` files; the archive and the restored bytes a seeded sample of at most `max_bytes`
    positions (restored ones inside the files only: the gaps of the output are never written).  At most 44 MB."""
    torch, dev = rt.cx.torch, rt.cx.dev

    def sample(count, k):
        return np.sort(np.random.default_rng(seed).choice(count, size=min(count, k), replace=False))

    def take(t, idx):
        return t[torch.from_numpy(idx.astype(np.int64)).to(dev)].cpu().numpy()

    files = sample(rt.n, max_files)
    entries = sample(rt.u_n, max_files)
    nb = int(rt.nbytes[0])
    arch_pos = np.sort(np.random.default_rng(seed).integers(0, nb, size=min(nb, max_bytes)))
    lens = rt.mine.len.astype(np.int64)
    ends = np.cumsum(lens)
    pos = np.sort(np.random.default_rng(seed).integers(0, rt.B, size=min(rt.B, max_bytes)))
    f = np.searchsorted(ends, pos, side="right")
    out_pos = rt.mine.off.astype(np.int64)[f] + pos - (ends[f] - lens[f])
    arrays = {
        "pack_digests": take(rt.d_dig[: rt.n * 32].view(rt.n, 32), files).astype(np.float32),
        "pack_first": take(rt.d_first, files).astype(np.float32),
        "pack_frame_offset": take(rt.d_foff, files).astype(np.float64),
        "pack_frame_length": take(rt.d_flen, files).astype(np.float64),
        "pack_frames_bytes": np.array([nb], dtype=np.float64),
        "pack_frames_sample": take(rt.d_frames, arch_pos).astype(np.float32),
        "unpack_ok": take(rt.d_ok, entries).astype(np.float32),
        "unpack_status": take(rt.d_status, entries).astype(np.float64),
        "unpack_out_sample": take(rt.d_out, out_pos).astype(np.float32),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def leg_roundtrip(cx: Ctx, glob, level: int, steps: int, warmup: int, checksum: bool = True, partition: str = "auto"):
    """One corpus shape, pack + unpack device-resident -> dict for `extras`."""
    rt = RoundTrip(cx, glob, level, checksum=checksum, partition=partition)
    try:
        ms, tp, tu = time_roundtrip(cx, rt, steps, warmup)
        Btot = cx.rank_sum(float(rt.B))
        Utot = cx.rank_sum(float(rt.u_bytes))
        uniq = cx.rank_sum(float((rt.ln * rt.d_first[: rt.n].to(cx.torch.int64)).sum().item()))
        Ctot = cx.rank_sum(float(rt.nbytes[0]))
        return {"files": int(cx.rank_sum(float(rt.n))), "bytes": Btot, "unique_bytes": uniq, "compressed_bytes": Ctot, "ratio": uniq / max(Ctot, 1.0),
                "pack_ms": tp, "unpack_ms": tu, "pack_gbs": Btot / tp / 1e6, "unpack_gbs": Utot / tu / 1e6,
                "roundtrip_gbs": Btot / ms / 1e6, "steps": steps, "warmup": warmup, "checksum": checksum, "rank0_step_ms": rt.step_ms,
                "partition": "contiguous" if rt.plan.contiguous else "greedy", "roundtrip_verified": True}
    finally:
        rt.free()


def leg_c5(cx: Ctx, produced, args, steps: int):
    """Unpack + BLAKE3 verify of reference-made frames, per level.  `produced` = c5_produce() of this rank's share."""
    from zarc_b200 import corpus

    torch, lib = cx.torch, cx.lib
    out = {}
    unique = None
    for level, P in produced.items():
        U = int(P["ulen"].sum())
        R = max(1, int(round(args.c5_total_gb * 1e9 / len(produced) / cx.world / max(U, 1))))
        A = int(P["archive"].shape[0])
        K = int(P["len"].shape[0])
        d_arch = cx.to_dev(P["archive"]).repeat(R)
        off_r = np.concatenate([P["off"] + np.uint64(r * A) for r in range(R)])
        d_off, d_len, d_ul = cx.to_dev(off_r.astype(np.int64)), cx.to_dev(np.tile(P["len"], R).astype(np.int64)), cx.to_dev(np.tile(P["ulen"], R).astype(np.int64))
        ul_r = np.tile(P["ulen"], R)
        d_oo = cx.to_dev((np.cumsum(ul_r) - ul_r).astype(np.int64))
        d_dig = cx.to_dev(np.tile(P["digests"], R))
        total = U * R
        d_out = torch.empty(total + 64, dtype=torch.uint8, device=cx.dev)
        d_ok = torch.zeros(K * R, dtype=torch.uint8, device=cx.dev)
        d_st = torch.zeros(K * R, dtype=torch.int32, device=cx.dev)
        dctx = lib.zg_dctx_create()
        lib.check(lib.zg_dctx_set_stream(dctx, cx.stream))

        def run():
            lib.check(lib.zg_unpack_batch_dev(dctx, d_arch.data_ptr(), A * R, K * R, d_off.data_ptr(), d_len.data_ptr(), d_ul.data_ptr(), d_dig.data_ptr(),
                                              d_out.data_ptr(), total, d_oo.data_ptr(), d_ok.data_ptr(), d_st.data_ptr()))

        run()
        cx.sync_all()
        ok = int(d_ok.sum().item()) == K * R and int(d_st.abs().sum().item()) == 0
        # byte-identical: the first and the last replica against the mix regenerated on the device (same file order)
        if unique is None:
            mix = corpus.c5_mix(total_bytes=int(args.c5_unique_gb * 1e9), seed=5)
            sub = corpus.take(mix, P["idx"], name="C5-mix shard")
            so, sl, sk, key = sub.segments()
            ublob = torch.empty(sub.blob_bytes + 64, dtype=torch.uint8, device=cx.dev)
            segs = [cx.to_dev(x) for x in (so, sl, sk, key)]
            lib.check(lib.zg_corpus_generate_dev(cx.stream, ublob.data_ptr(), *[t.data_ptr() for t in segs], len(so)))
            torch.cuda.synchronize()
            pieces = [ublob[int(o) : int(o) + int(l)] for o, l in zip(sub.off, sub.len)]
            unique = torch.cat(pieces) if pieces else ublob[:0]
            del ublob, pieces, segs
        same = all(bool(torch.equal(d_out[b + o : b + min(U, o + (1 << 30))], unique[o : min(U, o + (1 << 30))]))
                   for b in (0, (R - 1) * U) for o in range(0, U, 1 << 30))
        stats = (C.c_uint64 * 3)()
        lib.dll.zg_internal_decode_stats(stats)
        t = []
        for _ in range(steps):
            a, b = cx.ev(), cx.ev()
            cx.sync_all()
            a.record()
            run()
            b.record()
            cx.sync_all()
            t.append(cx.rank_max(a.elapsed_time(b)))
        ms = sum(t) / len(t)
        Ntot, Ctot = cx.rank_sum(float(total)), cx.rank_sum(float(A * R))
        cpu_unpack = cx.rank_max(P["cpu_unpack_s"])
        cpu_pack = cx.rank_max(P["cpu_pack_s"])
        Uall = cx.rank_sum(float(U))
        out[f"L{level}"] = {"frames": int(cx.rank_sum(float(K * R))), "unique_bytes": Uall, "replication": R, "bytes": Ntot, "compressed_bytes": Ctot,
                            "ratio_reference": Ntot / max(Ctot, 1.0), "unpack_verify_ms": ms, "unpack_verify_gbs": Ntot / ms / 1e6,
                            "byte_identical": same, "all_digests_verified": ok,
                            "decode_stats": {"frames": int(stats[0]), "work_items": int(stats[1]), "frames_decoded_twice": int(stats[2])},
                            "cpu_reference": {"unpack_verify_gbs": Uall / cpu_unpack / 1e9, "pack_gbs": Uall / cpu_pack / 1e9,
                                              "cores": args.cpu_cores_used, "what": "oracle/ref_path.py on the same files (one process per core)"}}
        lib.zg_dctx_free(dctx)
        del d_arch, d_out, d_off, d_len, d_ul, d_oo, d_dig, d_ok, d_st
        torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="c2 only: corpus-gb per GPU (weak) or in total (strong)")
    ap.add_argument("--partition", default="auto", choices=["auto", "greedy", "contiguous"])
    ap.add_argument("--extras", default="auto", help="auto (config c2: strong,c4,c3,c5) | none | comma list of strong,c1,c3,c4,c5,nocksum")
    ap.add_argument("--corpus-gb", type=float, default=10.2, help="C2: uncompressed GB per GPU (10.2 GB = ~1M files)")
    ap.add_argument("--e2e-gb", type=float, default=0.0, help="GB per GPU through the host-buffer ABI per e2e step (0: the whole shard)")
    ap.add_argument("--c3-files", type=int, default=8)
    ap.add_argument("--c3-file-gib", type=float, default=4.0)
    ap.add_argument("--c4-gb", type=float, default=20.0)
    ap.add_argument("--c5-unique-gb", type=float, default=2.2, help="unique input per level the reference path compresses on the host")
    ap.add_argument("--c5-total-gb", type=float, default=50.0, help="total decoded bytes per unpack pass over the three levels (replication on device)")
    ap.add_argument("--level", type=int, default=3)
    ap.add_argument("--levels-sample-gb", type=float, default=0.5, help="C2 sample packed at levels 1/3/9 for the ratio table")
    ap.add_argument("--cpu-sample-mb-per-core", type=float, default=96.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (a seeded sample) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "ours" or args.config == "c5" or world > 1):
        ap.error("--dump-outputs needs --impl ours, one GPU and a pack + unpack config (c1-c4)")
    cores = host_cores()
    my_cores = max(1, cores // world)
    args.cpu_cores_used = my_cores * world
    workload = workload_text(args.config, args, world, args.scaling)
    extras_on = []
    if args.extras == "auto":
        extras_on = (["strong"] if world > 1 else []) + ["levels", "c4", "c3", "nocksum", "c5"] if args.config == "c2" else []
    elif args.extras != "none":
        extras_on = [x for x in args.extras.split(",") if x]

    # -------------------------------------------------------------------------------------------
    # the helper libraries of the host-side legs (workload generator, C oracle) are built here, once per process, not by
    # every forked worker at the same time (the builds themselves are atomic: temp file + rename)
    from oracle import ref_path as _rp
    from zarc_b200 import build as _build

    _build.build_corpus_host()
    _rp.build_c_oracle()
    if args.impl == "reference":
        if rank != 0:
            return
        per_core = min(args.cpu_sample_mb_per_core, 48.0)
        sample = int(per_core * 1e6 * cores)
        for _ in range(args.warmup):
            cpu_reference_run(2, min(sample, int(8e6) * cores), args.level, cores)
        vals = []
        t0 = time.perf_counter()
        for _ in range(args.steps):
            vals.append(cpu_reference_run(2, sample, args.level, cores))
        dt = time.perf_counter() - t0
        v = sum(x["bytes"] for x in vals) / sum(x["pack_s"] + x["unpack_s"] for x in vals) / 1e9
        sample_desc = (f"each step = {sample / 1e6:.0f} MB ({per_core:g} MB per core) of the C2 corpus the GPU arm packs in full, split over {cores} "
                       "processes; libzstd 1.5.5 + BLAKE3 with the reference's call sequence (oracle/ref_path.py), in memory, no file I/O; "
                       "the corpus generator is tools/libzarc_corpus.so (the product library is not loaded)")
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / max(args.steps, 1) * 1e3, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_text("c2", args, args.gpus, args.scaling), "sample_bytes_per_step": sample, "sample": sample_desc},
            "pack_gbs": float(np.mean([x["pack_gbs"] for x in vals])), "unpack_gbs": float(np.mean([x["unpack_gbs"] for x in vals])),
            "ratio": float(np.mean([x["ratio"] for x in vals])),
            "cpu_baseline": {"value": v, "unit": "GB/s", "cores": cores, "kind": "port", "sample": sample_desc},
            "e2e": {"value": v, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    # -------------------------------------------------------------------------------------------
    # host-side work first (fork before CUDA is initialised): CPU baseline (rank 0, N=1) and the C5 producer.
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.config == "c2":
        sample = int(args.cpu_sample_mb_per_core * 1e6 * cores)
        cpu = cpu_reference_run(2, sample, args.level, cores)
        cpu["sample"] = (f"{sample / 1e6:.0f} MB of the same C2 corpus, split over {cores} processes; libzstd 1.5.5 + BLAKE3 with the "
                         "reference's call sequence (oracle/ref_path.py), in memory, no file I/O")
    ref_ratios = None
    if rank == 0 and "levels" in extras_on:
        try:
            ref_ratios = cpu_ratio_run(2, int(args.levels_sample_gb * 1e9), (1, 3, 9), cores)
        except Exception as e:
            ref_ratios = {"error": f"{type(e).__name__}: {e}"}
    c5 = None
    c5_err = None
    if args.config == "c5" or "c5" in extras_on:
        try:
            # every rank produces the frames of its own share of the mix with its share of the host cores
            t0 = time.perf_counter()
            full = c5_produce(5, int(args.c5_unique_gb * 1e9), (1, 3, 9), cores) if world == 1 else None
            if world > 1:
                # shard = every world-th worker slice: run nworkers = my_cores * world virtual workers, keep mine
                import multiprocessing as mp

                nw = my_cores * world
                ctx = mp.get_context("fork")
                with ctx.Pool(my_cores) as pool:
                    res = pool.map(_c5_worker, [(5, int(args.c5_unique_gb * 1e9), (1, 3, 9), w, nw) for w in range(rank, nw, world)])
                full = {}
                idx = np.concatenate([r[0] for r in res])
                ulen = np.concatenate([r[1] for r in res])
                dig = np.frombuffer(b"".join(r[2] for r in res), dtype=np.uint8)
                for level in (1, 3, 9):
                    flen = np.concatenate([r[3][level][1] for r in res])
                    full[level] = dict(archive=np.frombuffer(b"".join(r[3][level][0] for r in res), dtype=np.uint8), len=flen,
                                       off=(np.cumsum(flen) - flen).astype(np.uint64), ulen=ulen, digests=dig, idx=idx,
                                       cpu_pack_s=max(r[3][level][2] for r in res), cpu_unpack_s=max(r[3][level][3] for r in res))
            c5 = full
            c5_host_s = time.perf_counter() - t0
        except Exception as e:  # the headline must not depend on an extra
            c5_err = f"{type(e).__name__}: {e}"

    import torch
    import torch.distributed as dist

    from zarc_b200 import corpus, lib as product_lib

    torch.cuda.set_device(local_rank)
    lib = product_lib()
    assert lib.zg_device_count() > 0, "no CUDA device"
    lib.check(lib.zg_set_device(local_rank))
    # rank 0's stdout carries exactly one JSON line: NCCL (version banner) and anything else that writes to fd 1 from
    # native code goes to stderr; the line itself is written to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/zarc_bench_nccl.%h.%p.log")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cx = Ctx(lib, torch, dist, rank, world, local_rank)
    dev, stream = cx.dev, cx.stream
    if os.environ.get("ZG_DECODE_BATCHING"):  # tuning aid: "cap_div,min_batch_bytes,floor_bytes"
        a, b, c3 = os.environ["ZG_DECODE_BATCHING"].split(",")
        lib.dll.zg_internal_set_decode_batching(C.c_uint32(int(a)), C.c_uint32(int(b)), C.c_uint32(int(c3)))
    if os.environ.get("ZG_CHAIN_MODE"):  # tuning aid: 0 per-block flags, 1 chain executor when the frames fit, 2 always
        lib.dll.zg_internal_set_decode_chain_mode(C.c_uint32(int(os.environ["ZG_CHAIN_MODE"])))
    if os.environ.get("ZG_SLICE_MB"):  # tuning aid: host-API slice size
        lib.dll.zg_internal_set_slice_bytes(C.c_uint64(int(os.environ["ZG_SLICE_MB"]) << 20))
    if os.environ.get("ZG_UNPACK_WORKERS"):  # tuning aid: slices decoded at the same time by the host API
        lib.dll.zg_internal_set_unpack_workers(C.c_int(int(os.environ["ZG_UNPACK_WORKERS"])))
    if os.environ.get("ZG_PACK_SLICE_MB"):  # tuning aid: host-API slice size, pack only
        lib.dll.zg_internal_set_pack_slice_bytes(C.c_uint64(int(os.environ["ZG_PACK_SLICE_MB"]) << 20))

    def shape(config, scaling=args.scaling):
        if config == "c2":
            return corpus.c2_source_tree(total_bytes=int(args.corpus_gb * 1e9) * (world if scaling == "weak" else 1), seed=2)
        if config == "c1":
            return corpus.c1_tree()
        if config == "c3":
            return corpus.c3_huge(n_files=args.c3_files, file_bytes=int(args.c3_file_gib * (1 << 30)))
        if config == "c4":
            return corpus.c2_source_tree(total_bytes=int(args.c4_gb * 1e9), seed=4, dup=True)
        raise ValueError(config)

    # -------------------------------------------------------------------------------------------
    # the line's own workload
    line = {"metric": METRIC, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
            "scaling": args.scaling if args.config == "c2" else "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic"}
    launches0 = lib.zg_kernel_launch_count()
    sampler = ClockSampler(local_rank)
    if args.config == "c5":
        assert c5 is not None, c5_err
        if rank == 0:
            sampler.start()
            time.sleep(0.3)
        r5 = leg_c5(cx, c5, args, max(args.steps, 1))
        clocks = sampler.stop() if rank == 0 else None
        Ntot = sum(v["bytes"] for v in r5.values())
        ms = sum(v["unpack_verify_ms"] for v in r5.values())
        line.update({"metric": "unpack+verify GB/s (uncompressed) of reference-made frames", "value": Ntot / ms / 1e6, "ms_per_step": ms,
                     "config": {"workload": workload, "l2": "inputs (>= 10x L2) larger than L2; no flush needed"}, "levels": r5,
                     "gpu_launches": int(lib.zg_kernel_launch_count() - launches0), "clocks": clocks, "c5_host_seconds": c5_host_s})
        if rank == 0:
            os.write(json_fd, (json.dumps(line) + "\n").encode())
        if world > 1:
            dist.destroy_process_group()
        return

    rt = RoundTrip(cx, shape(args.config), args.level, partition=args.partition)
    n, B = rt.n, rt.B
    for i in range(args.warmup):
        rt.pack()
        if i == 0:
            rt.prepare_unpack()
        rt.unpack()
    cx.sync_all()
    rt.verify()  # correctness of what is being timed: digests verified on device, bytes identical
    uniq_bytes = float((rt.ln * rt.d_first[:n].to(torch.int64)).sum().item())
    ratio = uniq_bytes / max(float(rt.nbytes[0]), 1.0)

    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    lib.zg_profile_enable(1)
    launches0 = lib.zg_kernel_launch_count()
    cx.sync_all()
    e0, e1 = cx.ev(), cx.ev()
    pack_ms, unpack_ms = [], []
    e0.record()
    for _ in range(args.steps):
        a, b, c = cx.ev(), cx.ev(), cx.ev()
        a.record()
        rt.pack()
        b.record()
        rt.unpack()
        c.record()
        pack_ms.append((a, b))
        unpack_ms.append((b, c))
    e1.record()
    cx.sync_all()
    total_ms = e0.elapsed_time(e1)
    launches = lib.zg_kernel_launch_count() - launches0
    lib.zg_profile_enable(0)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(rt, args.dump_outputs)
    tp = sum(x.elapsed_time(y) for x, y in pack_ms) / args.steps
    tu = sum(x.elapsed_time(y) for x, y in unpack_ms) / args.steps
    step_ms = {"pack": [round(x.elapsed_time(y), 2) for x, y in pack_ms], "unpack": [round(x.elapsed_time(y), 2) for x, y in unpack_ms]}
    if rt.host_ms:
        step_ms["pack_host_parts[digests,dedup_exchange,encode,offsets_exchange]"] = rt.host_ms[-args.steps:]
    total_ms = cx.rank_max(total_ms)
    tp, tu = cx.rank_max(tp), cx.rank_max(tu)
    Btot = cx.rank_sum(float(B))
    ms_per_step = total_ms / args.steps
    value = Btot / (ms_per_step * 1e-3) / 1e9

    # per-kernel roofline of the dominant kernel (device time from CUDA events on the launching stream)
    prof = {}
    names = ((0, "k_blake3_chunks"), (6, "k_zstd_match_blocks"), (7, "k_zstd_literals"), (8, "k_zstd_sequences"), (2, "k_zstd_decode_frames"),
             (1, "encode pass (match+literals+sequences, all chunks)"))
    for k, name in names:
        ms, cnt = C.c_double(0), C.c_uint64(0)
        lib.zg_profile_read(k, C.byref(ms), C.byref(cnt))
        prof[name] = (ms.value, cnt.value)
    peak, peak_src = measured_peaks()
    C_bytes = float(rt.nbytes[0])
    # algorithmic bytes per STEP of each kernel class (SURVEY.md 8d): the encoder reads the unique input once (match) and
    # writes the compressed bytes once (literals + sequences sections); the decoder reads C and writes N; BLAKE3 reads N
    # (pack digests and unpack verification: two launches per step)
    alg_step = {"k_blake3_chunks": 2.0 * B, "k_zstd_match_blocks": uniq_bytes, "k_zstd_literals": C_bytes, "k_zstd_sequences": C_bytes,
                "k_zstd_decode_frames": C_bytes + B, "encode pass (match+literals+sequences, all chunks)": uniq_bytes + C_bytes}
    single = [nm for _, nm in names[:5]]
    dom = max(single, key=lambda k: prof[k][0])
    kernels = {}
    for k, v in prof.items():
        ms_step = v[0] / args.steps
        kernels[k] = {"ms_per_step": ms_step, "launches_per_step": v[1] / args.steps,
                      "ms_per_launch": (v[0] / v[1] if v[1] else None),
                      "algorithmic_gbs": (alg_step[k] / (ms_step * 1e-3) / 1e9 if ms_step > 0 else None),
                      "share_of_step": (ms_step / ms_per_step if ms_per_step else None)}
    lps = max(prof[dom][1] / args.steps, 1)
    dom_ms = prof[dom][0] / max(prof[dom][1], 1)
    alg_launch = alg_step[dom] / lps
    achieved = alg_launch / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    roofline = {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic(dom, (uniq_bytes if dom != "k_zstd_decode_frames" else float(B)) / lps), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_launch, "kernels": kernels,
                "note": "integer/latency-bound kernels (bitstream decode, match finding, entropy coding); the HBM roofline is the "
                        "ceiling the north star names for decode and verify; BLAKE3 and match finding are bound by INT32 issue "
                        "(int_issue below: this repo's measured INT32 peak, tools/kbench.py --what intpeak)"}
    isp = os.path.join(ROOT, "profiles", "ncu_issue.json")
    if os.path.exists(isp):
        try:
            I = json.load(open(isp))
            roofline["issue"] = {"what": "issue-slot utilisation of the hot kernels from the committed ncu captures: the ceiling that applies to the "
                                         "latency-bound kernels (match finding, entropy coding, decoding)",
                                 **{k: v for k, v in I.items() if not k.startswith("_")}}
        except Exception:
            pass
    ip = os.path.join(ROOT, "profiles", "int_peak.json")
    if os.path.exists(ip):
        try:
            P = json.load(open(ip))
            lane_ops = float(P["int32_lane_ops_per_s"])
            b3 = kernels["k_blake3_chunks"]["algorithmic_gbs"]
            roofline["int_issue"] = {
                "peak_int32_lane_ops_per_s": lane_ops, "peak_source": P.get("how"),
                "k_blake3_chunks": {"bound": "int_issue", "ops_per_byte": 13.1, "ceiling_gbs": lane_ops / 13.1 / 1e9,
                                   "achieved_gbs": b3, "frac": (b3 / (lane_ops / 13.1 / 1e9)) if b3 else None, "hbm_frac": (b3 / peak) if b3 else None},
            }
        except Exception:
            pass

    # -------------------------------------------------------------------------------------------
    # end to end through the host-buffer C ABI (pinned host memory, copies inside the timed region)
    e2e = None
    if not args.no_e2e:
        import psutil

        want = B if args.e2e_gb <= 0 else min(B, int(args.e2e_gb * 1e9))
        # pinned: input + frames + output ~ 3.3 x the shard; stay inside half of this rank's share of the free host memory
        room = int(psutil.virtual_memory().available * 0.5 / world / 3.3)
        want = max(1, min(want, room))
        sub = rt.mine.subset(max(1, int(n * min(1.0, want / max(B, 1)))))
        ne, Be, span = sub.n_files, sub.total_bytes, sub.blob_bytes
        h_blob = torch.empty(span + 64, dtype=torch.uint8, pin_memory=True)
        h_blob[:span].copy_(rt.blob[:span])
        torch.cuda.synchronize()
        cap_e = Be + max(1024, Be // 10) + 32 * ne
        h_frames = torch.empty(cap_e, dtype=torch.uint8, pin_memory=True)
        h_out = torch.empty(Be + 64, dtype=torch.uint8, pin_memory=True)
        h_dig = torch.empty(ne * 32, dtype=torch.uint8, pin_memory=True)
        h_first = torch.empty(ne, dtype=torch.uint8, pin_memory=True)
        h_foff = torch.empty(ne, dtype=torch.int64, pin_memory=True)
        h_flen = torch.empty(ne, dtype=torch.int64, pin_memory=True)
        h_ok = torch.empty(ne, dtype=torch.uint8, pin_memory=True)
        h_status = torch.empty(ne, dtype=torch.int32, pin_memory=True)
        h_off = torch.from_numpy(sub.off.astype(np.int64)).pin_memory()
        h_len = torch.from_numpy(sub.len.astype(np.int64)).pin_memory()
        nb_e = np.zeros(1, dtype=np.uint64)
        cctx, dctx = rt.cctx, rt.dctx
        e2e_t = [0.0, 0.0]
        e2e_steps = []

        def e2e_step():
            t0 = time.perf_counter()
            lib.check(lib.zg_cctx_reset_archive(cctx, 12))
            lib.check(lib.zg_pack_batch(cctx, h_blob.data_ptr(), h_off.data_ptr(), h_len.data_ptr(), ne, h_dig.data_ptr(), h_first.data_ptr(),
                                        h_foff.data_ptr(), h_flen.data_ptr(), h_frames.data_ptr(), cap_e, nb_e.ctypes.data))
            t1 = time.perf_counter()
            rel = h_foff - 12
            lib.check(lib.zg_unpack_batch(dctx, h_frames.data_ptr(), int(nb_e[0]), ne, rel.data_ptr(), h_flen.data_ptr(), h_len.data_ptr(),
                                          h_dig.data_ptr(), h_out.data_ptr(), Be, None, h_ok.data_ptr(), h_status.data_ptr()))
            t2 = time.perf_counter()
            e2e_t[0] += t1 - t0  # both calls return with their results on the host (blocking API)
            e2e_t[1] += t2 - t1
            e2e_steps.append([round((t1 - t0) * 1e3, 1), round((t2 - t1) * 1e3, 1)])

        for _ in range(2):
            e2e_step()
        cx.sync_all()
        assert int(h_ok.sum().item()) == ne, "e2e verification failed"
        s0, s1 = cx.ev(), cx.ev()
        ksteps = max(2, min(args.steps, 5))
        e2e_t[0] = e2e_t[1] = 0.0
        e2e_steps.clear()
        s0.record()
        for _ in range(ksteps):
            e2e_step()
        s1.record()
        cx.sync_all()
        e_ms = cx.rank_max(s0.elapsed_time(s1)) / ksteps
        Ce = float(nb_e[0])
        e2e = {"value": cx.rank_sum(float(Be)) / (e_ms * 1e-3) / 1e9, "unit": "GB/s",
               "h2d_bytes_per_step": int(span + 16 * ne + Ce + 56 * ne), "d2h_bytes_per_step": int(Ce + 49 * ne + Be + 5 * ne),
               "ms_per_step": e_ms, "pack_ms": e2e_t[0] / ksteps * 1e3, "unpack_ms": e2e_t[1] / ksteps * 1e3,
               "rank0_step_ms_pack_unpack": list(e2e_steps), "workload_gb_per_gpu": Be / 1e9, "whole_shard": bool(ne == n),
               "api": "zg_pack_batch + zg_unpack_batch (host buffers, pinned), digests verified"}
        # the host link of THIS box, measured on the same pinned buffers right after the timed steps (tools/linkbench.py's
        # method: 1 GiB per direction, all ranks released together, slowest rank's device time; boxes differ by 10-30 %)
        live = None
        try:
            nb = min(1 << 30, span, Be)
            d_a = torch.empty(nb, dtype=torch.uint8, device=dev)
            d_b = torch.empty(nb, dtype=torch.uint8, device=dev)
            s2 = torch.cuda.Stream()

            def _h2d():
                d_a.copy_(h_blob[:nb], non_blocking=True)

            def _d2h():
                h_out[:nb].copy_(d_b, non_blocking=True)

            def _both():
                s2.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s2):
                    h_out[:nb].copy_(d_b, non_blocking=True)
                d_a.copy_(h_blob[:nb], non_blocking=True)
                torch.cuda.current_stream().wait_stream(s2)

            live = {}
            for name, fn in (("h2d_gbs", _h2d), ("d2h_gbs", _d2h), ("duplex_each_way_gbs", _both)):
                fn()
                best = 1e30
                for _ in range(3):
                    cx.sync_all()
                    a, b = cx.ev(), cx.ev()
                    a.record()
                    for _ in range(2):
                        fn()
                    b.record()
                    torch.cuda.synchronize()
                    best = min(best, cx.rank_max(a.elapsed_time(b)))
                live[name] = world * 2 * nb / best / 1e6
            del d_a, d_b
        except Exception as e:
            live = {"error": f"{type(e).__name__}: {e}"}
        lp = os.path.join(ROOT, "profiles", "host_link.json")
        if live and "duplex_each_way_gbs" in live:
            # one step moves max(h2d, d2h) bytes per rank each way; the link runs both ways at once
            ceil_ms = max(e2e["h2d_bytes_per_step"], e2e["d2h_bytes_per_step"]) * world / (live["duplex_each_way_gbs"] * 1e6)
            # pack is an upload with a smaller download beside it, unpack the reverse: the two calls run one after the
            # other, so the step cannot be shorter than each call's larger direction at that direction's own rate
            serial_ms = (span * world / (live["h2d_gbs"] * 1e6)) + (Be * world / (live["d2h_gbs"] * 1e6))
            e2e["link_ceiling"] = {"aggregate_duplex_gbs_each_way": live["duplex_each_way_gbs"], "h2d_gbs": live["h2d_gbs"], "d2h_gbs": live["d2h_gbs"],
                                   "ms_per_step_at_ceiling": ceil_ms, "frac_of_ceiling": ceil_ms / e_ms,
                                   "ms_per_step_pack_upload_plus_unpack_download": serial_ms, "frac_of_serial_bound": serial_ms / e_ms,
                                   "source": "measured in this run on the e2e's own pinned buffers (1 GiB per direction, all ranks at once, "
                                             "slowest rank's CUDA-event time), right after the timed steps"}
        elif os.path.exists(lp):
            try:
                L = json.load(open(lp))
                key = str(world)
                if key in L.get("aggregate_duplex_gbs_each_way", {}):
                    # one step moves max(h2d, d2h) bytes per rank each way; the link runs both ways at once
                    ceil_ms = max(e2e["h2d_bytes_per_step"], e2e["d2h_bytes_per_step"]) * world / (L["aggregate_duplex_gbs_each_way"][key] * 1e6)
                    e2e["link_ceiling"] = {"aggregate_duplex_gbs_each_way": L["aggregate_duplex_gbs_each_way"][key], "ms_per_step_at_ceiling": ceil_ms,
                                           "frac_of_ceiling": ceil_ms / e_ms, "source": L.get("how")}
            except Exception:
                pass
        del h_blob, h_frames, h_out

    files_total = int(cx.rank_sum(float(n)))
    part = "contiguous byte-balanced ranges" if rt.plan.contiguous else "size-balanced greedy deal"
    rt.free()
    del rt

    # -------------------------------------------------------------------------------------------
    # the other BASELINE.json shapes, as extras of the same line (each leg verified; a failing leg reports its error)
    extras = {}
    ex_steps = 2

    def leg(name, fn):
        t0 = time.perf_counter()
        try:
            extras[name] = fn()
            extras[name]["wall_s"] = time.perf_counter() - t0
        except Exception as e:
            extras[name] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()

    if "levels" in extras_on:
        # ratio (and pack rate) at levels 1 / 3 / 9 next to libzstd's on the same C2 sample (north star: "the compression
        # ratio at each level is reported next to the reference's")
        def levels_leg():
            sample = corpus.c2_source_tree(total_bytes=int(args.levels_sample_gb * 1e9), seed=2)
            out = {}
            for lv in (1, 3, 9):
                r = leg_roundtrip(cx, sample, lv, 2, 2)
                ref = ref_ratios.get(lv) if isinstance(ref_ratios, dict) else None
                out[f"L{lv}"] = {"ratio": r["ratio"], "ratio_reference": ref, "ours_over_reference_size": (ref / r["ratio"]) if ref else None,
                                 "pack_gbs": r["pack_gbs"], "unpack_gbs": r["unpack_gbs"]}
            out["sample"] = f"{args.levels_sample_gb:g} GB of the C2 corpus (seed 2), the same files for both"
            return out

        leg("levels", levels_leg)
    if "strong" in extras_on and world > 1:
        leg("c2_strong", lambda: dict(leg_roundtrip(cx, shape("c2", "strong"), args.level, max(2, min(args.steps, 5)), 2),
                                      workload=workload_text("c2", args, world, "strong")))
    if "c4" in extras_on:
        leg("c4", lambda: dict(leg_roundtrip(cx, shape("c4"), args.level, ex_steps, 1), workload=workload_text("c4", args, world, "strong")))
    if "c1" in extras_on:
        leg("c1", lambda: dict(leg_roundtrip(cx, shape("c1"), args.level, ex_steps, 1), workload=workload_text("c1", args, world, "strong")))
    if "c3" in extras_on:
        leg("c3", lambda: dict(leg_roundtrip(cx, shape("c3"), args.level, 1, 1), workload=workload_text("c3", args, world, "strong")))
    if "nocksum" in extras_on:
        leg("c3_checksum_off", lambda: dict(leg_roundtrip(cx, shape("c3"), args.level, 1, 1, checksum=False),
                                            workload=workload_text("c3", args, world, "strong") + " with ChecksumFlag(false) (pack.rs:92)"))
    if "c5" in extras_on:
        if c5 is None:
            extras["c5"] = {"error": c5_err}
        else:
            leg("c5", lambda: {"levels": leg_c5(cx, c5, args, 2), "workload": workload_text("c5", args, world, "strong"), "host_produce_s": c5_host_s})

    if rank == 0:
        line.update({
            "value": value, "ms_per_step": ms_per_step,
            "config": {"workload": workload, "files_per_gpu": n, "bytes_per_gpu": B, "files_total": files_total,
                       "l2": "inputs (>= 10x L2) larger than L2; no flush needed",
                       "parallelism": f"files sharded over {world} GPU(s) by {part}; per step: NCCL all-gather of digests (global dedup) and of frame sizes (archive offsets)"
                       if world > 1 else "1 GPU"},
            "pack_gbs": Btot / (tp * 1e-3) / 1e9, "unpack_gbs": Btot / (tu * 1e-3) / 1e9,
            "ratio": ratio, "ratio_reference_level3": cpu["ratio"] if cpu else None, "rank0_step_ms": step_ms,
            "roofline": roofline,
            "cpu_baseline": ({"value": cpu["value"], "unit": "GB/s", "cores": cores, "kind": "port", "sample": cpu["sample"],
                              "pack_gbs": cpu["pack_gbs"], "unpack_gbs": cpu["unpack_gbs"]} if cpu else None),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "extras": extras,
        })
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

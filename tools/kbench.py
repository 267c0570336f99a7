"""Per-kernel device-resident micro-benchmarks (CUDA events on the launching stream)."""
import argparse
import json
import sys
import os
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from zarc_b200 import lib as product_lib, corpus  # noqa: E402


def dev(a):
    return torch.from_numpy(a).cuda()


def gen_corpus(lib, c, stream=0):
    so, sl, sk, key = c.segments()
    blob = torch.empty(max(c.blob_bytes, 1) + 64, dtype=torch.uint8, device="cuda")
    d = [dev(x) for x in (so, sl, sk, key)]
    lib.check(lib.zg_corpus_generate_dev(stream, blob.data_ptr(), d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), len(so)))
    torch.cuda.synchronize()
    return blob


def timeit(fn, iters=5, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return min(ts), sorted(ts)[len(ts) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=2.0)
    ap.add_argument("--what", default="blake3,xxh64")
    ap.add_argument("--sample-mb", type=float, default=100)
    ap.add_argument("--replicas", type=int, default=10)
    ap.add_argument("--level", type=int, default=3)
    args = ap.parse_args()
    lib = product_lib()
    res = {}
    import ctypes as C

    if os.environ.get("ZG_DECODE_SHARE"):  # tuning aid: first batches = 4 / q of a warp's fair share of the frames
        lib.dll.zg_internal_set_decode_share(C.c_uint32(int(os.environ["ZG_DECODE_SHARE"])))
    if os.environ.get("ZG_DECODE_BATCHING"):  # tuning aid: "cap_div,min_batch_bytes,floor_bytes" (zstd_decode.cu: the hand-out)
        import ctypes as C

        a, b, c3 = os.environ["ZG_DECODE_BATCHING"].split(",")
        lib.dll.zg_internal_set_decode_batching(C.c_uint32(int(a)), C.c_uint32(int(b)), C.c_uint32(int(c3)))
    if os.environ.get("ZG_ENC_CHUNK_MB"):  # tuning aid: input bytes per encoder chunk (zstd_encode.cu)
        import ctypes as C

        lib.dll.zg_internal_set_encode_chunk_bytes(C.c_uint64(int(os.environ["ZG_ENC_CHUNK_MB"]) << 20))
    if os.environ.get("ZG_B3_VARIANT"):  # tuning aid: staging / arithmetic variant of k_blake3_chunks (blake3.cu: b3c_launch)
        lib.dll.zg_internal_set_b3_variant(int(os.environ["ZG_B3_VARIANT"]))
    c = corpus.c2_source_tree(total_bytes=int(args.gb * 1e9))
    t0 = time.time()
    blob = gen_corpus(lib, c)
    res["gen_s"] = time.time() - t0
    off, ln = dev(c.off), dev(c.len)
    n = c.n_files
    s = torch.cuda.current_stream().cuda_stream
    if "intpeak" in args.what:
        import ctypes as C

        f = lib.dll.zg_internal_int_peak
        f.restype = C.c_size_t
        f.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        peak = {}
        for mode, name in enumerate(["iadd3", "lop3", "shf", "prmt", "blake3_g_mix"]):
            best = 0.0
            for ctas in (4, 8):
                for _ in range(3):
                    ms, th, ops = C.c_double(0), C.c_uint64(0), C.c_uint64(0)
                    lib.check(f(s, mode, 20000, ctas, C.byref(ms), C.byref(th), C.byref(ops)))
                    best = max(best, th.value * ops.value / (ms.value * 1e-3))
            peak[name] = best
        res["int_peak_lane_ops_per_s"] = peak
        sm = torch.cuda.get_device_properties(0).multi_processor_count
        res["int_peak_lane_ops_per_clk_per_sm_at_1965MHz"] = {k: v / sm / 1.965e9 for k, v in peak.items()}
        json.dump({"int32_lane_ops_per_s": peak["blake3_g_mix"], "single_op_lane_instr_per_s": {k: peak[k] for k in ("iadd3", "lop3", "shf", "prmt")},
                   "sms": sm,
                   "how": "tools/kbench.py --what intpeak: zarc_b200/csrc/peak.cu, 8 independent chains per thread, 256 threads x 4-8 CTAs per SM, "
                          "best of 3, CUDA events; the figure used as the INT32 roofline is the BLAKE3 quarter-round mix (add3 / xor / rotates by "
                          "16 and 12), operations counted as SURVEY.md App. B counts BLAKE3's 792 per compression"},
                  open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "int_peak.json"), "w"))
    if "pcie" in args.what:
        # host link: pinned copies, each direction alone and both at once (what bounds the e2e number)
        nb = 1 << 30
        hb, hb2 = torch.empty(nb, dtype=torch.uint8, pin_memory=True), torch.empty(nb, dtype=torch.uint8, pin_memory=True)
        db, db2 = torch.empty(nb, dtype=torch.uint8, device="cuda"), torch.empty(nb, dtype=torch.uint8, device="cuda")
        s2 = torch.cuda.Stream()
        best, _ = timeit(lambda: db.copy_(hb, non_blocking=True), iters=5, warmup=2)
        res["pcie_h2d_gbs"] = nb / best / 1e6
        best, _ = timeit(lambda: hb.copy_(db, non_blocking=True), iters=5, warmup=2)
        res["pcie_d2h_gbs"] = nb / best / 1e6

        def both():
            s2.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s2):
                hb2.copy_(db2, non_blocking=True)
            db.copy_(hb, non_blocking=True)
            torch.cuda.current_stream().wait_stream(s2)

        best, _ = timeit(both, iters=5, warmup=2)
        res["pcie_duplex_gbs_each"] = nb / best / 1e6
        del hb, hb2, db, db2
    if "blake3" in args.what:
        dig = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
        best, med = timeit(lambda: lib.check(lib.zg_blake3_batch_dev(s, blob.data_ptr(), off.data_ptr(), ln.data_ptr(), n, dig.data_ptr())))
        res["blake3_c2_gbs"] = c.total_bytes / best / 1e6
        if os.environ.get("ZG_B3_SWEEP"):
            for v in range(13):
                lib.dll.zg_internal_set_b3_variant(v)
                best, med = timeit(lambda: lib.check(lib.zg_blake3_batch_dev(s, blob.data_ptr(), off.data_ptr(), ln.data_ptr(), n, dig.data_ptr())))
                res[f"blake3_c2_gbs_variant{v}"] = c.total_bytes / best / 1e6
            lib.dll.zg_internal_set_b3_variant(int(os.environ.get("ZG_B3_VARIANT", "9")))
        c3 = corpus.c3_huge(n_files=4, file_bytes=512 << 20)
        b3 = gen_corpus(lib, c3)
        o3, l3 = dev(c3.off), dev(c3.len)
        d3 = torch.empty(4 * 32, dtype=torch.uint8, device="cuda")
        best, med = timeit(lambda: lib.check(lib.zg_blake3_batch_dev(s, b3.data_ptr(), o3.data_ptr(), l3.data_ptr(), 4, d3.data_ptr())))
        res["blake3_c3_gbs"] = c3.total_bytes / best / 1e6
        del b3
    if "xxh64" in args.what:
        h = torch.empty(n, dtype=torch.int64, device="cuda")
        best, med = timeit(lambda: lib.check(lib.zg_xxh64_batch_dev(s, blob.data_ptr(), off.data_ptr(), ln.data_ptr(), n, h.data_ptr())))
        res["xxh64_c2_gbs"] = c.total_bytes / best / 1e6
        c3 = corpus.c3_huge(n_files=4, file_bytes=512 << 20)
        b3 = gen_corpus(lib, c3)
        o3, l3 = dev(c3.off), dev(c3.len)
        h3 = torch.empty(4, dtype=torch.int64, device="cuda")
        best, med = timeit(lambda: lib.check(lib.zg_xxh64_batch_dev(s, b3.data_ptr(), o3.data_ptr(), l3.data_ptr(), 4, h3.data_ptr())), iters=3, warmup=1)
        res["xxh64_c3_gbs_per_file"] = c3.total_bytes / 4 / best / 1e6
        del b3
    if "decode" in args.what:
        from oracle import ref_path
        import concurrent.futures as cf

        cs = corpus.c2_source_tree(total_bytes=int(args.sample_mb * 1e6), seed=5)
        hblob = corpus.materialise_host(lib, cs)
        datas = [bytes(hblob[int(o) : int(o) + int(l)]) for o, l in zip(cs.off, cs.len)]
        t0 = time.time()
        frames = [ref_path.ref_compress(d, level=args.level) for d in datas]
        res["ref_compress_gbs_1core"] = cs.total_bytes / (time.time() - t0) / 1e9
        res["ref_ratio"] = cs.total_bytes / sum(len(f) for f in frames)
        arch = np.frombuffer(b"".join(frames), dtype=np.uint8)
        flen = np.array([len(f) for f in frames], dtype=np.uint64)
        foff = (np.cumsum(flen) - flen).astype(np.uint64)
        R = args.replicas
        A = len(arch)
        d_arch = dev(arch).repeat(R)
        off_r = np.concatenate([foff + np.uint64(r * A) for r in range(R)])
        len_r = np.tile(flen, R)
        ul_r = np.tile(cs.len, R)
        oo_r = (np.cumsum(ul_r) - ul_r).astype(np.uint64)
        total = int(ul_r.sum())
        d_out = torch.empty(total + 64, dtype=torch.uint8, device="cuda")
        d_off, d_len, d_ul, d_oo = dev(off_r), dev(len_r), dev(ul_r), dev(oo_r)
        K = len(off_r)
        d_status = torch.zeros(K, dtype=torch.int32, device="cuda")
        dctx = lib.zg_dctx_create()
        lib.zg_dctx_set_stream(dctx, s)
        for vc in (0, 1):
            lib.zg_dctx_set_verify_checksum(dctx, vc)
            best, med = timeit(lambda: lib.check(lib.zg_unpack_batch_dev(dctx, d_arch.data_ptr(), A * R, K, d_off.data_ptr(), d_len.data_ptr(),
                               d_ul.data_ptr(), None, d_out.data_ptr(), total, d_oo.data_ptr(), None, d_status.data_ptr())), iters=3, warmup=1)
            res[f"decode_c2_L{args.level}_gbs_ck{vc}"] = total / best / 1e6
        # check the bytes of replica 0 and the last replica
        ho = d_out[: cs.total_bytes].cpu().numpy().tobytes()
        res["decode_ok"] = ho == b"".join(datas) and int(d_status.abs().sum()) == 0
        res["decode_total_gb"] = total / 1e9
        # + BLAKE3 verify
        dig = np.frombuffer(b"".join(__import__("blake3").blake3(d).digest() for d in datas), dtype=np.uint8)
        d_dig = dev(np.tile(dig, R))
        d_ok = torch.zeros(K, dtype=torch.uint8, device="cuda")
        best, med = timeit(lambda: lib.check(lib.zg_unpack_batch_dev(dctx, d_arch.data_ptr(), A * R, K, d_off.data_ptr(), d_len.data_ptr(),
                           d_ul.data_ptr(), d_dig.data_ptr(), d_out.data_ptr(), total, d_oo.data_ptr(), d_ok.data_ptr(), d_status.data_ptr())), iters=3, warmup=1)
        res[f"unpack_verify_c2_L{args.level}_gbs"] = total / best / 1e6
        res["verify_all_ok"] = int(d_ok.sum()) == K
        lib.zg_dctx_free(dctx)
    if "pack" in args.what:
        cctx = lib.zg_cctx_create()
        lib.zg_cctx_set_stream(cctx, s)
        lib.check(lib.zg_cctx_init(cctx, 0))
        lib.check(lib.zg_cctx_set_parameter(cctx, 201, 1))
        lib.check(lib.zg_cctx_set_parameter(cctx, 100, args.level))
        cap = c.total_bytes + c.total_bytes // 10 + 64 * n
        d_dig = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
        d_first = torch.empty(n, dtype=torch.uint8, device="cuda")
        d_foff = torch.empty(n, dtype=torch.int64, device="cuda")
        d_flen = torch.empty(n, dtype=torch.int64, device="cuda")
        d_frames = torch.empty(cap, dtype=torch.uint8, device="cuda")
        nbytes = np.zeros(1, dtype=np.uint64)

        def run_pack():
            lib.check(lib.zg_cctx_reset_archive(cctx, 12))
            lib.check(lib.zg_pack_batch_dev(cctx, blob.data_ptr(), off.data_ptr(), ln.data_ptr(), n, d_dig.data_ptr(), d_first.data_ptr(),
                                            d_foff.data_ptr(), d_flen.data_ptr(), d_frames.data_ptr(), cap, nbytes.ctypes.data))

        lib.zg_profile_enable(1)
        best, med = timeit(run_pack, iters=3, warmup=1)
        lib.zg_profile_enable(0)
        import ctypes as C
        for k, name in enumerate(["blake3", "encode", "decode", "assemble", "xxh64", "dedup", "match", "literals", "sequences"]):
            ms, cnt = C.c_double(0), C.c_uint64(0)
            lib.zg_profile_read(k, C.byref(ms), C.byref(cnt))
            if cnt.value:
                res[f"ms_{name}"] = round(ms.value / cnt.value, 3)
        res[f"pack_c2_L{args.level}_gbs"] = c.total_bytes / best / 1e6
        res["pack_ratio"] = c.total_bytes / float(nbytes[0])
        res["pack_unique"] = int(d_first.sum())
        # unpack what we packed
        dctx = lib.zg_dctx_create()
        lib.zg_dctx_set_stream(dctx, s)
        d_out = torch.empty(c.blob_bytes + 64, dtype=torch.uint8, device="cuda")
        d_ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        d_status = torch.zeros(n, dtype=torch.int32, device="cuda")
        d_foff0 = d_foff - 12

        def run_unpack():
            lib.check(lib.zg_unpack_batch_dev(dctx, d_frames.data_ptr(), int(nbytes[0]), n, d_foff0.data_ptr(), d_flen.data_ptr(), ln.data_ptr(),
                                              d_dig.data_ptr(), d_out.data_ptr(), c.blob_bytes, off.data_ptr(), d_ok.data_ptr(), d_status.data_ptr()))

        lib.zg_profile_enable(1)
        best, med = timeit(run_unpack, iters=3, warmup=1)
        lib.zg_profile_enable(0)
        for k, name in ((0, "blake3_verify"), (2, "decode"), (9, "huf_literals")):
            ms, cnt = C.c_double(0), C.c_uint64(0)
            lib.zg_profile_read(k, C.byref(ms), C.byref(cnt))
            if cnt.value:
                res[f"ms_{name}"] = round(ms.value / cnt.value, 3)
        res["unpack_ms"] = round(best, 3)
        res[f"unpack_own_c2_gbs"] = c.total_bytes / best / 1e6
        res["roundtrip_ok"] = bool(int(d_ok.sum()) == n and torch.equal(d_out[: c.blob_bytes], blob[: c.blob_bytes]))
        lib.zg_cctx_free(cctx)
        lib.zg_dctx_free(dctx)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

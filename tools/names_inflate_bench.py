"""Device Inflate of the identifiers slices (idn_gpu_inflate_names) against the host's zlib inflate.

    python tools/names_inflate_bench.py [--reads 5368704] [--file-reads 10000000] [--sweep] [--out result.json]

1. the codec alone: blocks of 41 943 reads (bench.py's workload blocks), 32 blocks per call as the host mirror makes them,
   slices written by zlib level 6 and by the device encoder (idn_gpu_deflate_names); host zlib inflate on all cores (one
   block per task, as inflate_names) against idn_gpu_inflate_names + fetch (the call uploads the slices itself: ~3.5 MB
   per call of bench titles).  Wall clock around calls that end in a device synchronise, one warm-up pass, best of 3;
   GB/s of name bytes; the stats of the parallel decode (chunks joined, bytes decoded serially).
2. e2e_file-shaped decompress with identifiers: .idn -> FASTQ text through the host mirror's text path (FastqTextReader,
   two contexts on the device, thread_num = cores), names inflated by the host and by the device, alternated, two passes.
3. --sweep: the codec-alone leg on zlib-6 bench titles over ranges of 4 to 64 KiB (idn_gpu_set_inflate_range).
Prints one JSON object (and writes it to --out)."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
import zlib
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from names_deflate_bench import CALL_BLOCKS, PER_BLOCK, bench_titles, fastq_text, gpu_info, illumina  # noqa: E402


def z6(x):
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    return c.compress(x) + c.flush()


def inflate_raw(x):
    d = zlib.decompressobj(-15)
    return d.decompress(x)


def slices(ctx, names, off, codec):
    """per call: (payload, block_off, block_first_read), the joined names of its blocks"""
    n = len(off) - 1
    calls = []
    for r0 in range(0, n, PER_BLOCK * CALL_BLOCKS):
        r1 = min(n, r0 + PER_BLOCK * CALL_BLOCKS)
        bf = (np.append(np.arange(r0, r1, PER_BLOCK), r1) - r0).astype(np.uint32)
        if codec == "zlib6":
            texts = []
            for b in range(len(bf) - 1):
                a, e = int(bf[b]) + r0, int(bf[b + 1]) + r0
                rel = (off[a:e + 1] - off[a]).astype(np.int64)
                texts.append(np.insert(names[int(off[a]):int(off[e])], rel[1:-1], 10).tobytes())
            with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
                zs = list(ex.map(z6, texts))
            recs = [b"\x00" + len(z).to_bytes(4, "big") + b"\x01" + z for z in zs]
            payload = b"".join(recs)
            bo = np.zeros(len(recs) + 1, dtype=np.uint64)
            bo[1:] = np.cumsum([len(r) for r in recs])
        else:
            o = (off[r0:r1 + 1] - off[r0]).astype(np.uint64)
            out, bo = ctx.deflate_names(o, names[int(off[r0]):int(off[r1])], bf)
            payload = out.tobytes()
        calls.append((np.frombuffer(payload, dtype=np.uint8), bo, bf))
    return calls


def codec_alone(ctx, names, off, label, codec):
    calls = slices(ctx, names, off, codec)
    name_bytes = int(off[-1])
    stats = []

    def dev_pass():
        stats.clear()
        for payload, bo, bf in calls:
            _, _, st = ctx.inflate_names(payload, bo, bf)
            stats.append(st)

    def host_pass(ex):
        jobs = []
        for payload, bo, _ in calls:
            for b in range(len(bo) - 1):
                p = payload[int(bo[b]):int(bo[b + 1])].tobytes()
                jobs.append(p[6:])
        return sum(len(t) for t in ex.map(inflate_raw, jobs))

    dev_pass()
    t_dev = []
    for _ in range(3):
        t0 = time.perf_counter()
        dev_pass()
        t_dev.append(time.perf_counter() - t0)
    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        host_pass(ex)
        t_host = []
        for _ in range(3):
            t0 = time.perf_counter()
            host_pass(ex)
            t_host.append(time.perf_counter() - t0)
    tot = {k: sum(s[k] for s in stats) for k in stats[0]}
    return {"names": label, "slices_by": codec, "reads": len(off) - 1, "name_bytes": name_bytes, "calls": len(calls),
            "slice_bytes": tot["in_bytes"], "device_GBps_of_name_bytes": name_bytes / min(t_dev) / 1e9, "device_pass_s": t_dev,
            f"host_zlib_{os.cpu_count()}_threads_GBps": name_bytes / min(t_host) / 1e9, "host_pass_s": t_host, "stats": tot}


def e2e_file(torch, host, n_reads):
    text = fastq_text(n_reads)
    models = [host.Model.load(ROOT / "models" / "SRR8861483__human__illumina_novaseq_6000__acids.msgpack"),
              host.Model.load(ROOT / "models" / "SRR8861483__human__illumina_novaseq_6000__q_scores.msgpack")]
    cores = os.cpu_count() or 1
    c = host.IdnCompressor(models, thread_num=cores, devices=[0, 0])
    c.add_fastq_text(text)
    idn = np.frombuffer(c.finish(), dtype=np.uint8)
    c.close()
    back_h = torch.empty(text.size + 64, dtype=torch.uint8, pin_memory=True).numpy()
    res = {"fastq_bytes": int(text.size), "reads": n_reads, "container_bytes": int(idn.size), "thread_num": cores,
           "contexts_on_the_device": 2}
    runs = {False: [], True: []}
    for it in range(3):  # pass 0 warms up both
        for on_dev in (False, True):
            t0 = time.perf_counter()
            n = 0
            for v in host.FastqTextReader(models, idn, devices=[0, 0], thread_num=cores, identifiers_on_device=on_dev):
                back_h[n:n + v.size] = v
                n += v.size
            t1 = time.perf_counter()
            ok = n == text.size and bool(np.array_equal(back_h[:n], text))
            if it:
                runs[on_dev].append({"decompress_GBps": text.size / (t1 - t0) / 1e9, "round_trip": ok})
    res["host_inflate"] = runs[False]
    res["device_inflate"] = runs[True]
    host.release_cached()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4 * CALL_BLOCKS * PER_BLOCK, help="bench titles for the codec-alone leg")
    ap.add_argument("--illumina-reads", type=int, default=CALL_BLOCKS * PER_BLOCK)
    ap.add_argument("--file-reads", type=int, default=10_000_000, help="reads of the e2e_file-shaped leg (0 = skip)")
    ap.add_argument("--sweep", action="store_true", help="range-size sweep on zlib-6 bench titles")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from idencomp_b200 import capi, host
    ctx = capi.Context(0)
    res = {"gpu": gpu_info()}
    bt, ill = bench_titles(a.reads), illumina(a.illumina_reads)
    res["codec_alone"] = [codec_alone(ctx, *bt, "bench titles r%012d 1:N:0", "zlib6"),
                          codec_alone(ctx, *bt, "bench titles r%012d 1:N:0", "device"),
                          codec_alone(ctx, *ill, "Illumina-like", "zlib6"),
                          codec_alone(ctx, *ill, "Illumina-like", "device")]
    print(json.dumps(res, indent=1), flush=True)
    if a.sweep:
        sw = []
        small = (bt[0][:int(bt[1][CALL_BLOCKS * PER_BLOCK])], bt[1][:CALL_BLOCKS * PER_BLOCK + 1])
        for r in (4096, 8192, 16384, 32768, 65536):
            ctx.set_inflate_range(r)
            row = codec_alone(ctx, *small, "bench titles r%012d 1:N:0", "zlib6")
            sw.append({"range": r, "device_GBps_of_name_bytes": row["device_GBps_of_name_bytes"], "stats": row["stats"]})
        ctx.set_inflate_range(4096)
        res["range_sweep"] = sw
        print(json.dumps(sw, indent=1), flush=True)
    ctx.close()
    if a.file_reads:
        res["e2e_file"] = e2e_file(torch, host, a.file_reads)
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(s + "\n")


if __name__ == "__main__":
    main()

"""Device Deflate of the identifiers slice (idn_gpu_deflate_names_dev) against the host's zlib level 6.

    python tools/names_deflate_bench.py [--reads 40500000] [--file-reads 20000000] [--out result.json]

1. the codec alone: names on the device, blocks of 41 943 reads (bench.py's workload blocks), one call per 32 blocks as the
   host mirror makes them; wall clock around calls that end in a device synchronise, after a warm-up pass; GB/s of name
   bytes, and the Deflate bytes beside zlib-6 on the same blocks.  Bench titles `r%012d 1:N:0` and Illumina-like names.
2. e2e_file-shaped: FASTQ text in page-locked memory -> .idn -> FASTQ text through the host mirror, two contexts on the
   device, thread_num = cores, identifiers by the host's zlib and by the device codec, alternated, two passes each.
Prints one JSON object (and writes it to --out)."""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import time
import zlib
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

PER_BLOCK = 41_943
CALL_BLOCKS = 32


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def bench_titles(n):
    idx = np.arange(n, dtype=np.int64)
    digits = np.stack([(idx // 10 ** k) % 10 for k in range(11, -1, -1)], axis=1).astype(np.uint8) + 48
    head = np.full((n, 1), ord("r"), dtype=np.uint8)
    tail = np.broadcast_to(np.frombuffer(b" 1:N:0", dtype=np.uint8), (n, 6))
    names = np.concatenate([head, digits, tail], axis=1).reshape(-1)
    return names, np.arange(n + 1, dtype=np.uint64) * 19


def illumina(n, seed=1):
    rng = random.Random(seed)
    x = y = 1000
    out = []
    for _ in range(n):
        x += rng.randint(1, 40)
        if x > 32000:
            x = 1000
            y += rng.randint(1, 300)
        out.append(b"A00123:8:H5TJ3DSXX:1:1101:%d:%d 1:N:0:ACGTACGT+TTGCAGGA" % (x, y))
    off = np.zeros(n + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(s) for s in out])
    return np.frombuffer(b"".join(out), dtype=np.uint8), off


def codec_alone(torch, capi, ctx, names, off, label):
    n = len(off) - 1
    dev = torch.device("cuda", 0)
    names_d = torch.from_numpy(names.copy()).to(dev)
    calls = []
    for r0 in range(0, n, PER_BLOCK * CALL_BLOCKS):
        r1 = min(n, r0 + PER_BLOCK * CALL_BLOCKS)
        bf = np.append(np.arange(r0, r1, PER_BLOCK), r1).astype(np.uint32) - r0
        calls.append((r0, torch.from_numpy(bf.view(np.int32)).to(dev), len(bf) - 1, int(off[r1] - off[r0]), r1 - r0))
    cap = max(int(ctx.L.idn_gpu_deflate_names_bound(nb_, nr, len(bf) - 1)) for _, bf, _, nb_, nr in calls)
    out_d = torch.empty(cap, dtype=torch.uint8, device=dev)
    so_d = torch.empty(CALL_BLOCKS + 1, dtype=torch.int64, device=dev)
    # per call: names of its reads, its own name_off (rebased) and blocks
    offs = [torch.from_numpy((off[r0:r0 + nr + 1] - off[r0]).view(np.int64)).to(dev) for r0, _, _, _, nr in calls]

    def one_pass():
        total = 0
        for (r0, bf_d, nb, _, nr), o_d in zip(calls, offs):
            base = names_d[int(off[r0]):]
            ctx.check(ctx.L.idn_gpu_deflate_names_dev(ctx.h, base.data_ptr(), o_d.data_ptr(), bf_d.data_ptr(), nb, out_d.data_ptr(), cap,
                                                      so_d.data_ptr(), None))
            torch.cuda.synchronize()
            so = so_d[:nb + 1].cpu().numpy()
            total += int(so[-1]) - 6 * nb
        return total

    z_dev = one_pass()  # warm-up, and the Deflate bytes for the ratio
    times = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        one_pass()
        times.append(time.perf_counter() - t0)
    blocks = []
    for r0, bf_d, nb, _, nr in calls:
        bf = bf_d.cpu().numpy().astype(np.int64) + r0
        for b in range(nb):
            a, e = off[bf[b]], off[bf[b + 1]]
            rel = (off[bf[b]:bf[b + 1] + 1] - a).astype(np.int64)
            blocks.append(np.insert(names[a:e], rel[1:-1], 10).tobytes())

    def z6(x):
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        return len(c.compress(x) + c.flush())

    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        z_host = sum(ex.map(z6, blocks))
    t0 = time.perf_counter()
    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        list(ex.map(z6, blocks))
    t_host = time.perf_counter() - t0
    joined = sum(len(b) for b in blocks)
    return {"names": label, "reads": n, "name_bytes": int(off[-1]), "blocks": len(blocks),
            "device_GBps_of_name_bytes": int(off[-1]) / min(times) / 1e9, "device_pass_s": times,
            "device_bytes_per_joined_byte": z_dev / joined, "zlib6_bytes_per_joined_byte": z_host / joined,
            "device_over_zlib6": z_dev / z_host, f"host_zlib6_{os.cpu_count()}_threads_GBps": int(off[-1]) / t_host / 1e9}


def fastq_text(n, read_len=100, seed=7):
    rng = np.random.default_rng(seed)
    names, _ = bench_titles(n)
    rec = np.empty((n, 1 + 19 + 1 + read_len + 3 + read_len + 1), dtype=np.uint8)
    rec[:, 0] = ord("@")
    rec[:, 1:20] = names.reshape(n, 19)
    rec[:, 20] = 10
    rec[:, 21:21 + read_len] = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=(n, read_len))]
    p = 21 + read_len
    rec[:, p:p + 3] = np.frombuffer(b"\n+\n", dtype=np.uint8)
    rec[:, p + 3:p + 3 + read_len] = rng.integers(35, 75, size=(n, read_len), dtype=np.uint8)
    rec[:, -1] = 10
    return rec.reshape(-1)


def e2e_file(torch, host, n_reads):
    text = fastq_text(n_reads)
    text_h = torch.empty(text.size, dtype=torch.uint8, pin_memory=True).numpy()
    text_h[:] = text
    del text
    models = [host.Model.load(ROOT / "models" / "SRR8861483__human__illumina_novaseq_6000__acids.msgpack"),
              host.Model.load(ROOT / "models" / "SRR8861483__human__illumina_novaseq_6000__q_scores.msgpack")]
    cores = os.cpu_count() or 1
    idn_h = torch.empty(text_h.size + (64 << 20), dtype=torch.uint8, pin_memory=True).numpy()  # random quality scores
    back_h = torch.empty(text_h.size + 64, dtype=torch.uint8, pin_memory=True).numpy()
    res = {"fastq_bytes": int(text_h.size), "reads": n_reads, "thread_num": cores, "contexts_on_the_device": 2}
    runs = {False: [], True: []}
    for it in range(3):  # pass 0 warms up both (contexts, page-locked buffers); passes 1, 2 are reported
        for on_dev in (False, True):
            c = host.IdnCompressor(models, thread_num=cores, devices=[0, 0], identifiers_on_device=on_dev)
            c.set_output(idn_h)
            t0 = time.perf_counter()
            c.add_fastq_text(text_h)
            c.finish(copy=False)
            t1 = time.perf_counter()
            n_idn = int(c.output_view().size)
            st = c.stats()
            c.close()
            t2 = time.perf_counter()
            n_back = host.decompress_text_into(models, idn_h[:n_idn], back_h, device=0, thread_num=cores)
            t3 = time.perf_counter()
            ok = n_back == text_h.size and bool(np.array_equal(back_h[:n_back], text_h))
            if it:
                runs[on_dev].append({"compress_GBps": text_h.size / (t1 - t0) / 1e9, "decompress_GBps": text_h.size / (t3 - t2) / 1e9,
                                     "container_bytes": n_idn, "identifier_bytes": st["out_identifier_bytes"], "round_trip": ok})
    res["host_zlib6"] = runs[False]
    res["device_deflate"] = runs[True]
    host.release_cached()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=40_500_000, help="bench titles for the codec-alone leg")
    ap.add_argument("--illumina-reads", type=int, default=24 * PER_BLOCK)
    ap.add_argument("--file-reads", type=int, default=20_000_000, help="reads of the e2e_file-shaped leg (0 = skip)")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from idencomp_b200 import capi, host
    ctx = capi.Context(0)
    res = {"gpu": gpu_info()}
    res["codec_alone"] = [codec_alone(torch, capi, ctx, *bench_titles(a.reads), "bench titles r%012d 1:N:0"),
                          codec_alone(torch, capi, ctx, *illumina(a.illumina_reads), "Illumina-like")]
    ctx.close()
    torch.cuda.empty_cache()
    print(json.dumps(res, indent=1), flush=True)
    if a.file_reads:
        res["e2e_file"] = e2e_file(torch, host, a.file_reads)
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(s + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- FASTQ compress/decompress throughput of the rANS hot path on B200 (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W            # this repository's CUDA path
    python bench.py --impl reference --gpus N ...            # the reference algorithm on the box's host cores

A step = one pass of the hot path over the workload's batch: compress every block, then decompress every block.
`value` = FASTQ text bytes through the codec per second (2 x FASTQ bytes / (t_compress + t_decompress)), inputs
resident in HBM, timed with CUDA events on the launching stream.  `e2e` = the same through the host-pointer C-ABI
calls (pinned host buffers, H2D/D2H inside the timed region; one context, one host thread, one self-pipelining call per
direction).  The same JSON line carries `workloads` (sub-records with value / e2e / roofline for the other named
configurations: NovaSeq-shaped 150 bp in the native format, PacBio-shaped long reads in both formats, per-read selection
among 4 + 4 models), `e2e_file` (FASTQ text -> .idn -> FASTQ text through the host mirror of the reference API, with and
without identifiers, and the identifiers codec alone), `fastq_text`, `other_mode` and, at N > 1, `strong_scaling` (ONE file
over the ranks).  --no-extra-workloads / --no-e2e / --no-fastq / --no-other-mode / --no-cpu-baseline trim the run.
--dump-outputs DIR writes what the last timed step of the headline workload handed back as DIR/<name>.npy (see
dump_outputs), so that two builds run with the same arguments can be compared output for output.
Nothing here reads /root/reference.
The oracle (oracle/) is used only for `cpu_baseline` / `--impl reference`: the Rust reference cannot be built in
this image, so its CPU restatement (pinned bit-exactly to the reference's golden container) is what is timed.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

MODELS = ROOT / "models"
BLOCK_SYMBOLS = 4 * 1024 * 1024  # IdnCompressorParams::max_block_total_len default, idn/compressor.rs:187
E2E_READS_PER_CALL = 16384       # e2e leg, native format: reads a sub-chunk of a host-pointer call should carry at least (PacBio-shaped sweep: 25 blocks 31.5, 50-64 blocks 44-48, 160-200 blocks 41.6-46 GB/s)
E2E_READS_PER_CALL_COMPAT = 32768  # compat format (a read is one serial chain): 59 blocks 31.7, 110-160 blocks 43, 320 blocks 41 GB/s (tools/r2_call_y.sh)

# SURVEY.md 8d.  fastq_overhead = bytes of a FASTQ record besides the 2*L symbol characters: '@' + name + '\n',
# '\n' after the acids, "+\n", '\n' after the quality scores.
WORKLOADS = {
    # config 2: 10 GB HiSeq 2000-shaped, 100 bp, compat mode.  The ERR174310 q-score model is missing from the
    # reference checkout (.MISSING_LARGE_BLOBS), SRR2962693 (same spec type, HiSeq 2500) stands in.
    "hiseq100": dict(acid="ERR174310__human__illumina_hiseq_2000__acids", q="SRR2962693__human__illumina_hiseq_2500__q_scores",
                     read_len=(100, 100), reads=40_485_830, name_len=41, seed=20240601, n_ppm=500, mode="compat", select=1,
                     desc="synthetic 10 GB Illumina HiSeq 2000-shaped FASTQ, 100 bp, compat mode (BASELINE.json configs[1])"),
    # config 3: 50 GB NovaSeq-shaped, 150 bp, native mode (142 857 143 reads x 350 B); a GPU that cannot hold it takes what fits
    "novaseq150_native": dict(acid="SRR8861483__human__illumina_novaseq_6000__acids", q="SRR8861483__human__illumina_novaseq_6000__q_scores",
                              read_len=(150, 150), reads=142_857_143, name_len=44, seed=20240602, n_ppm=500, mode="native", select=1,
                              desc="synthetic 50 GB NovaSeq 6000-shaped FASTQ, 150 bp, GPU-native multi-lane mode (BASELINE.json configs[2])"),
    # config 5: PacBio Sequel II-shaped long reads, variable-length blocks
    "pacbio": dict(acid="m64187e__sars_cov_2__sequel_ii_e__acids", q="m64187e__sars_cov_2__sequel_ii_e__q_scores",
                   read_len=(10_000, 20_000), reads=166_000, name_len=40, seed=20240603, n_ppm=0, mode="compat", select=1,
                   desc="synthetic 5 GB PacBio Sequel II-shaped FASTQ, 10-20 kb reads, compat mode (BASELINE.json configs[4])"),
    # the same long reads in the GPU-native format, which cuts them into lanes (a long read is many short chains there)
    "pacbio_native": dict(acid="m64187e__sars_cov_2__sequel_ii_e__acids", q="m64187e__sars_cov_2__sequel_ii_e__q_scores",
                          read_len=(10_000, 20_000), reads=166_000, name_len=40, seed=20240603, n_ppm=0, mode="native", select=1,
                          desc="synthetic 5 GB PacBio Sequel II-shaped FASTQ, 10-20 kb reads, GPU-native multi-lane mode (long reads cut into lanes)"),
    # configs[3] / the reference's default path: per-read greedy selection among the 4 + 4 models that quality 7 retains
    # (idn/compressor.rs:184-194, compressor_initializer.rs:53-74) out of the whole models/ directory
    "hiseq100_select4": dict(acid="ERR174310__human__illumina_hiseq_2000__acids", q="SRR2962693__human__illumina_hiseq_2500__q_scores",
                             read_len=(100, 100), reads=40_485_830, name_len=41, seed=20240601, n_ppm=500, mode="compat", select=4,
                             desc="synthetic 10 GB HiSeq-shaped FASTQ, 100 bp, compat mode, per-read model selection among the 4 + 4 "
                                  "models quality 7 retains from the 22 bundled ones (reference default path; BASELINE.json configs[3])"),
}
WORKLOADS["novaseq150"] = WORKLOADS["novaseq150_native"]  # round-1 name
EXTRA_WORKLOADS = ["novaseq150_native", "pacbio", "pacbio_native", "hiseq100_select4"]  # sub-records of the default run (the north-star shapes)


def read_lengths(w: dict, n_reads: int, first: int) -> np.ndarray:
    lo, hi = w["read_len"]
    if lo == hi:
        return np.full(n_reads, lo, dtype=np.uint64)
    rng = np.random.Generator(np.random.PCG64(w["seed"] + first))
    return rng.integers(lo, hi + 1, size=n_reads, dtype=np.uint64)


def form_blocks(lens: np.ndarray, max_len: int = BLOCK_SYMBOLS) -> np.ndarray:
    """IdnCompressor::add_sequence block forming (idn/compressor.rs:517-540) -> block_first_read."""
    if len(lens) and lens.min() == lens.max():
        per = max(1, max_len // int(lens[0]))
        first = np.arange(0, len(lens), per, dtype=np.uint32)
        return np.append(first, np.uint32(len(lens))).astype(np.uint32)
    first, cur = [0], 0
    for r, ln in enumerate(lens.tolist()):
        if cur + ln > max_len and cur > 0:
            first.append(r)
            cur = 0
        cur += ln
    first.append(len(lens))
    return np.asarray(first, dtype=np.uint32)


def fastq_bytes(w: dict, n_reads: int, n_symbols: int) -> int:
    return 2 * n_symbols + n_reads * (6 + w["name_len"])


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md).  The sampler is started ahead of the
    region (nvidia-smi takes a few hundred ms to deliver its first line, more with 8 ranks starting it at once) and only the
    samples whose own timestamps fall between begin() and end() count; a region shorter than the 100 ms period takes the
    nearest sample and says so."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def begin(self):
        import datetime
        self.t0 = datetime.datetime.now()

    def end(self):
        import datetime
        self.t1 = datetime.datetime.now()

    @staticmethod
    def parse(out: str):
        """[(timestamp or None, sm, sm_max, power, {reasons})] of the nvidia-smi lines"""
        import datetime
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for ln in out.splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f")
            except ValueError:
                ts = None
            try:
                row = (ts, float(f[2]), float(f[3]), float(f[4]), {n for n, v in zip(names, f[6:10]) if v.lower().startswith("active")})
            except ValueError:
                continue
            rows.append(row)
        return rows

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.t1 is None:
            self.end()
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=10)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        rows = self.parse(out)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        note = None
        if self.t0 is not None and all(r[0] is not None for r in rows):
            inside = [r for r in rows if self.t0 <= r[0] <= self.t1]
            if not inside:  # the region is shorter than the sampling period: the sample nearest to it
                mid = self.t0 + (self.t1 - self.t0) / 2
                near = min(rows, key=lambda r: abs((r[0] - mid).total_seconds()))
                off = min(abs((near[0] - self.t0).total_seconds()), abs((near[0] - self.t1).total_seconds()))
                note = f"no sample inside the {(self.t1 - self.t0).total_seconds() * 1e3:.0f} ms timed region: the nearest one, {off * 1e3:.0f} ms away"
                inside = [near]
            rows = inside
        res = {"sm_mhz": statistics.median(r[1] for r in rows), "sm_max_mhz": max(r[2] for r in rows), "power_w_max": max(r[3] for r in rows),
               "samples": len(rows), "reasons": sorted(set().union(*(r[4] for r in rows)))}
        if note:
            res["note"] = note
        return res


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle restatement) on the host cores
# ---------------------------------------------------------------------------------------------------------
def cpu_sample(w: dict, n_blocks: int, threads: int):
    from oracle import oracle as O
    am = O.Model(O.ModelData.load_msgpack(MODELS / (w["acid"] + ".msgpack")))
    qm = O.Model(O.ModelData.load_msgpack(MODELS / (w["q"] + ".msgpack")))
    lo, hi = w["read_len"]
    n_reads = max(1, int(n_blocks * BLOCK_SYMBOLS // ((lo + hi) // 2)))
    lens = read_lengths(w, n_reads, 0)
    ro = np.zeros(n_reads + 1, dtype=np.uint64)
    np.cumsum(lens, out=ro[1:])
    reads = O.synth_reads(am, qm, ro, 0, w["seed"], w["n_ppm"], threads=threads)
    return O, [am, qm], reads


def cpu_step(O, models, reads, threads: int):
    """compress + decompress once; returns (t_compress, t_decompress, container bytes)."""
    t0 = time.perf_counter()
    idn = O.compress(models, reads, max_block_total_len=BLOCK_SYMBOLS, include_identifiers=False, quality=7, fast=False,
                     threads=threads)
    t1 = time.perf_counter()
    back = O.decompress(models, idn, threads=threads)
    t2 = time.perf_counter()
    assert np.array_equal(back.acids, reads.acids) and np.array_equal(back.quals, reads.quals)
    return t1 - t0, t2 - t1, len(idn)


def run_reference(args, w: dict):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # bounded sample: two blocks per core keeps every worker busy; sized so K+W steps end within minutes
    n_blocks = args.cpu_blocks or max(8, min(2 * cores, 256))
    O, models, reads = cpu_sample(w, n_blocks, cores)
    fq = fastq_bytes(w, reads.n_reads, int(reads.read_off[-1]))
    for _ in range(args.warmup):
        cpu_step(O, models, reads, cores)
    tc = td = 0.0
    nbytes = 0
    for _ in range(args.steps):
        a, b, nbytes = cpu_step(O, models, reads, cores)
        tc += a
        td += b
    val = 2 * fq * args.steps / (tc + td) / 1e9
    sample = f"first {reads.n_reads} reads ({n_blocks} blocks, {fq / 1e6:.0f} MB FASTQ) of the workload per step"
    line = {
        "impl": "reference", "metric": "fastq_compress_decompress_GBps", "value": val, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": (tc + td) / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": w["desc"], "name": args.workload, "acid_model": w["acid"], "q_model": w["q"], "block_symbols": BLOCK_SYMBOLS,
                   "sample": sample},
        "compress_GBps": fq * args.steps / tc / 1e9, "decompress_GBps": fq * args.steps / td / 1e9,
        "container_bytes_per_read": nbytes / reads.n_reads,
        "cpu_baseline": {"value": val, "unit": "GB/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "reference-algorithm CPU restatement (oracle/), bit-identical to the reference's golden "
                                 "samples/1M.idn; the Rust reference cannot be built in this image (no rustc/cargo)"},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
class Chunk:
    __slots__ = ("r0", "r1", "b0", "b1", "s0", "s1", "n_reads", "n_syms", "n_blocks", "read_off", "block_first", "out_base",
                 "out_cap", "block_off", "block_crc", "stats", "dec_off", "dec_len", "dec_status", "dec_read_off", "batch")


class Env:
    """process-wide state of the GPU arm: device, torch, the library context, the process group"""
    pass


def setup_gpu():
    import torch

    from idencomp_b200 import capi, host
    env = Env()
    env.torch, env.capi, env.host = torch, capi, host
    env.rank = int(os.environ.get("RANK", "0"))
    env.world = int(os.environ.get("WORLD_SIZE", "1"))
    env.local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(env.local)
    env.dev = torch.device("cuda", env.local)
    env.dist = None
    if env.world > 1:
        import torch.distributed as dist
        # stdout carries the one JSON line and nothing else: NCCL's version banner (NCCL_DEBUG=VERSION/WARN on some boxes)
        # goes to stderr while the communicator is set up
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=env.dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
        env.dist = dist
    env.ctx = capi.Context(env.local)
    env.stream = torch.cuda.current_stream()
    env.sp = C.c_void_p(env.stream.cuda_stream)
    env.models = {}  # file stem -> (host.Model, handle in env.ctx)
    return env


def model_handle(env, stem: str) -> int:
    if stem not in env.models:
        m = env.host.Model.load(MODELS / (stem + ".msgpack"))
        env.models[stem] = (m, m.upload(env.ctx))
    return env.models[stem][1]


def retained_models(env, w: dict, block_reads: int):
    """The model set the reference's default path would code this workload with: IdnCompressor at quality 7 over the WHOLE
    models/ directory retains (7 + 1) / 2 = 4 models per type, clustered on the cost matrix of the first block
    (compressor_initializer.rs:53-74).  Runs the repository's host mirror (IdnCompressor, csrc/host/idn.cpp) on the first
    block of the workload; returns the file stems in container order (acid ids first)."""
    host, torch = env.host, env.torch
    ro = np.zeros(block_reads + 1, dtype=np.uint64)
    np.cumsum(read_lengths(w, block_reads, 0), out=ro[1:])
    S = int(ro[-1])
    a_d = torch.empty(S + 16, dtype=torch.uint8, device=env.dev)
    q_d = torch.empty(S + 16, dtype=torch.uint8, device=env.dev)
    ro_d = torch.from_numpy(ro.view(np.int64)).to(env.dev)
    env.ctx.check(env.ctx.L.idn_gpu_synth_reads_dev(env.ctx.h, model_handle(env, w["acid"]), model_handle(env, w["q"]), ro_d.data_ptr(),
                                                    block_reads, 0, w["seed"], w["n_ppm"], a_d.data_ptr(), q_d.data_ptr(), env.sp))
    torch.cuda.synchronize()
    stems = sorted(p.stem for p in MODELS.glob("*.msgpack"))
    all_models = [host.Model.load(MODELS / (st + ".msgpack")) for st in stems]
    by_id = {m.identifier: st for m, st in zip(all_models, stems)}
    c = host.IdnCompressor(all_models, quality=7, include_identifiers=False, device=env.local)
    c.add_batch(ro, a_d[:S].cpu().numpy(), q_d[:S].cpu().numpy())
    c.finish()
    names = [by_id[i] for i in c.retained_models()]
    c.close()
    return names


DUMP_SEED = 20240604
DUMP_SAMPLES = {"container": 4 << 20, "symbols": 2 << 20, "reads": 1 << 20}  # 40 MiB of samples at most


def _sample_positions(rng, n: int, k: int) -> np.ndarray:
    """k seeded positions in [0, n), ascending; all of them when n <= k"""
    return np.arange(n, dtype=np.int64) if n <= k else np.sort(rng.integers(0, n, size=k, dtype=np.int64))


def dump_outputs(out_dir: Path, chunks, out_d, dec_a, dec_q, S: int):
    """What the compress and decompress calls of the last timed step returned, as DIR/<name>.npy in float32 / float64
    (exact for bytes, CRCs and offsets below 2^53).  The whole outputs run to gigabytes, so the per-block tables are
    complete and the byte arrays are seeded samples (positions drawn from DUMP_SEED and the output's length):
      block_offsets       float64 [blocks + 1]  offset of every block in the concatenated container
      block_crc           float64 [blocks]      the CRC-32 the compressor returned for every block
      block_bytes_crc32   float64 [blocks]      CRC-32 of every block's container bytes (covers all of them)
      container_sample    float32               container bytes at sampled positions
      acids_sample        float32               decoded acids at sampled symbol positions
      quals_sample        float32               decoded quality scores at the same positions
      read_off_sample     float64               decoded read offsets at sampled read indices"""
    import zlib
    import torch
    rng = np.random.Generator(np.random.PCG64(DUMP_SEED))
    offs, crcs, digests, samples = [np.zeros(1, dtype=np.int64)], [], [], []
    base = 0
    block_off = [c.block_off.cpu().numpy() for c in chunks]
    total = sum(int(b[-1]) for b in block_off)
    pos = _sample_positions(rng, total, DUMP_SAMPLES["container"])
    for c, boff in zip(chunks, block_off):
        n = int(boff[-1])
        data = out_d[c.out_base:c.out_base + n].cpu().numpy()
        offs.append(base + boff[1:])
        crcs.append(c.block_crc.cpu().numpy().view(np.uint32))
        digests += [zlib.crc32(data[int(boff[b]):int(boff[b + 1])]) for b in range(c.n_blocks)]
        lo, hi = np.searchsorted(pos, [base, base + n])
        samples.append(data[pos[lo:hi] - base])
        base += n
    sym = torch.from_numpy(_sample_positions(rng, S, DUMP_SAMPLES["symbols"])).to(dec_a.device)
    read_off = torch.cat([c.dec_read_off[:-1] + c.s0 for c in chunks] + [torch.tensor([S], device=dec_a.device)])
    ridx = torch.from_numpy(_sample_positions(rng, len(read_off), DUMP_SAMPLES["reads"])).to(dec_a.device)
    arrays = {
        "block_offsets": np.concatenate(offs).astype(np.float64),
        "block_crc": np.concatenate(crcs).astype(np.float64),
        "block_bytes_crc32": np.asarray(digests, dtype=np.float64),
        "container_sample": np.concatenate(samples).astype(np.float32),
        "acids_sample": dec_a[sym].cpu().numpy().astype(np.float32),
        "quals_sample": dec_q[sym].cpu().numpy().astype(np.float32),
        "read_off_sample": read_off[ridx].cpu().numpy().astype(np.float64),
    }
    out_dir.mkdir(parents=True, exist_ok=True)
    for k, v in arrays.items():
        np.save(out_dir / f"{k}.npy", v)
    print(f"bench: {len(arrays)} output arrays ({sum(v.nbytes for v in arrays.values()) / 2**20:.1f} MiB) written to {out_dir}",
          file=sys.stderr)


def run_workload(env, args, name: str, w: dict, *, steps: int, warmup: int, main: bool, shard=None, no_e2e=False, after=None):
    """One workload on this rank's GPU: device-resident leg (timed with CUDA events), optional e2e leg (host buffers),
    and for the main workload the FASTQ text leg.  Returns the raw numbers of this rank; run_gpu reduces them over ranks."""
    torch, capi, ctx = env.torch, env.capi, env.ctx
    L, dev, sp, stream = ctx.L, env.dev, env.sp, env.stream
    rank, world = env.rank, env.world
    select = args.select if main and args.select > 1 else w.get("select", 1)

    # ---- the shard of this rank (weak scaling: every rank holds the workload's read count; strong scaling: `shard` =
    # (global index of the first read, reads) of this rank's contiguous block range of ONE file) ----
    n_reads = args.reads or w["reads"]
    lo, hi = w["read_len"]
    note = None
    if shard is not None:
        n_reads = shard[1]
    elif not (main and args.reads):
        # device memory of the device-resident leg per symbol: symbols in (2) + decoded out (2) + container capacity (1.5) and
        # ~1 more for the library's workspaces of a 1024-block call and the e2e staging
        free_b, _ = torch.cuda.mem_get_info()
        fit = int(0.80 * free_b / (6.5 * (lo + hi) / 2))
        if n_reads > fit and main and args.dump_outputs:  # a dump is only comparable with one of the same inputs
            raise SystemExit(f"{n_reads} reads asked, {fit} fit the free device memory: pass --reads to dump a fixed workload")
        if n_reads > fit:
            note = f"{n_reads} reads asked, {fit} fit the free device memory ({free_b / 1e9:.0f} GB)"
            n_reads = fit
    first_index = shard[0] if shard is not None else rank * n_reads
    lens = read_lengths(w, n_reads, first_index)
    read_off_h = np.zeros(n_reads + 1, dtype=np.uint64)
    np.cumsum(lens, out=read_off_h[1:])
    S = int(read_off_h[-1])
    block_first_h = form_blocks(lens)
    n_blocks = len(block_first_h) - 1
    fq = fastq_bytes(w, n_reads, S)

    model_names = [w["acid"], w["q"]]
    if select > 1:
        model_names = retained_models(env, w, int(block_first_h[1]))
        if w["acid"] not in model_names or w["q"] not in model_names:
            note = (note + "; " if note else "") + "the clustering did not retain the pair the reads were drawn from"
    handles = np.asarray([model_handle(env, st) for st in model_names], dtype=np.int32)
    n_handles = len(handles)

    read_off_d = torch.from_numpy(read_off_h.view(np.int64)).to(dev)
    acids_d = torch.empty(S + 16, dtype=torch.uint8, device=dev)
    quals_d = torch.empty(S + 16, dtype=torch.uint8, device=dev)
    ctx.check(L.idn_gpu_synth_reads_dev(ctx.h, model_handle(env, w["acid"]), model_handle(env, w["q"]), read_off_d.data_ptr(), n_reads,
                                        first_index, w["seed"], w["n_ppm"], acids_d.data_ptr(), quals_d.data_ptr(), sp))
    torch.cuda.synchronize()

    # ---- chunks of whole blocks: one library call per chunk and direction ----
    cb = args.chunk_blocks
    chunks = []
    out_total = 0
    for b0 in range(0, n_blocks, cb):
        c = Chunk()
        c.b0, c.b1 = b0, min(n_blocks, b0 + cb)
        c.r0, c.r1 = int(block_first_h[c.b0]), int(block_first_h[c.b1])
        c.s0, c.s1 = int(read_off_h[c.r0]), int(read_off_h[c.r1])
        c.n_reads, c.n_syms, c.n_blocks = c.r1 - c.r0, c.s1 - c.s0, c.b1 - c.b0
        c.read_off = torch.from_numpy((read_off_h[c.r0:c.r1 + 1] - read_off_h[c.r0]).view(np.int64)).to(dev)
        c.block_first = torch.from_numpy((block_first_h[c.b0:c.b1 + 1] - block_first_h[c.b0]).astype(np.int32)).to(dev)
        c.out_cap = int(L.idn_gpu_compress_bound(c.n_reads, c.n_syms, c.n_blocks, 0))
        if not args.full_bound:  # measured containers are ~0.35 B/symbol; 1.5 B/symbol + headers is ample and is checked
            c.out_cap = min(c.out_cap, int(1.5 * c.n_syms) + 21 * c.n_reads + 12 * c.n_blocks)
        c.out_base = out_total
        out_total += (c.out_cap + 255) // 256 * 256
        c.block_off = torch.zeros(c.n_blocks + 1, dtype=torch.int64, device=dev)
        c.block_crc = torch.zeros(c.n_blocks, dtype=torch.int32, device=dev)
        c.stats = torch.zeros(8, dtype=torch.int64, device=dev)
        c.dec_status = torch.zeros(4, dtype=torch.int32, device=dev)
        c.dec_read_off = torch.zeros(c.n_reads + 1, dtype=torch.int64, device=dev)
        b = capi.Batch()
        b.n_reads, b.n_symbols, b.n_blocks = c.n_reads, c.n_syms, c.n_blocks
        b.acids, b.quals = acids_d.data_ptr() + c.s0, quals_d.data_ptr() + c.s0
        b.read_off, b.block_first_read = c.read_off.data_ptr(), c.block_first.data_ptr()
        c.batch = b
        chunks.append(c)
    out_d = torch.empty(out_total + 16, dtype=torch.uint8, device=dev)
    dec_a = torch.empty(S + 16, dtype=torch.uint8, device=dev)
    dec_q = torch.empty(S + 16, dtype=torch.uint8, device=dev)

    MODES = {"compat": capi.MODE_COMPAT, "native": capi.MODE_NATIVE}
    if args.lane_symbols:
        ctx.set_lane_symbols(args.lane_symbols)

    def compress_all(mode):
        for c in chunks:
            ctx.check(L.idn_gpu_compress_blocks_dev(ctx.h, C.byref(c.batch), mode, handles.ctypes.data, n_handles, 0, None,
                                                    out_d.data_ptr() + c.out_base, c.out_cap, c.block_off.data_ptr(),
                                                    c.block_crc.data_ptr(), c.stats.data_ptr(), sp))

    def prepare_decode():
        """block table of the decode calls from the compress outputs (device ops, outside the timed region);
        returns ({chunk: container bytes}, container bytes, payload bytes)."""
        sizes, out_bytes, payload_bytes = {}, 0, 0
        for c in chunks:
            st = c.stats.cpu().numpy()
            if int(st[4]) > c.out_cap:
                raise SystemExit(f"container chunk needs {int(st[4])} bytes, capacity {c.out_cap}: rerun with --full-bound")
            c.dec_len = (c.block_off[1:] - c.block_off[:-1] - 8).to(torch.int32).contiguous()
            c.dec_off = torch.cat([c.block_off[:-1] + 8, c.block_off[-1:]]).contiguous()
            sizes[id(c)] = int(st[0])
            out_bytes += int(st[0])
            payload_bytes += int(st[3])
        return sizes, out_bytes, payload_bytes

    def decompress_all(mode, sizes):
        for c in chunks:
            ctx.check(L.idn_gpu_decompress_blocks_dev(ctx.h, out_d.data_ptr() + c.out_base, c.dec_off.data_ptr(),
                                                      c.dec_len.data_ptr(), c.block_crc.data_ptr(), c.n_blocks, sizes[id(c)],
                                                      mode, handles.ctypes.data, n_handles, dec_a.data_ptr() + c.s0,
                                                      dec_q.data_ptr() + c.s0, c.dec_read_off.data_ptr(), c.n_reads, c.n_syms,
                                                      c.dec_status.data_ptr(), sp))

    def check_decode_status():
        if os.environ.get("IDN_BENCH_NOVERIFY"):
            return
        for c in chunks:
            stt = c.dec_status.cpu().numpy()
            if int(stt[0]) != 0 or int(stt[2]) != c.n_reads:
                raise SystemExit(f"decode failed: status {stt.tolist()}")

    def barrier():
        torch.cuda.synchronize()
        if env.dist is not None:
            env.dist.barrier()
        torch.cuda.synchronize()

    def measure(mode_name, steps, warmup, profile):
        """W warm-up steps, then exactly `steps` timed steps with CUDA events on the launching stream."""
        mode = MODES[mode_name]
        compress_all(mode)
        torch.cuda.synchronize()
        sizes, out_bytes, payload_bytes = prepare_decode()
        dec_a.zero_()
        dec_q.zero_()
        decompress_all(mode, sizes)
        torch.cuda.synchronize()
        check_decode_status()
        sampler = ClockSampler(env.local)
        sampler.start()  # ahead of the timed region: only the samples stamped inside it count
        for _ in range(max(0, warmup - 1)):
            compress_all(mode)
            decompress_all(mode, sizes)
        barrier()
        if profile:
            ctx.profile(True)
        launches0 = ctx.launches
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        torch.cuda.synchronize()
        sampler.begin()
        t_wall0 = time.perf_counter()
        for k in range(steps):
            ev[k][0].record(stream)
            compress_all(mode)
            ev[k][1].record(stream)
            decompress_all(mode, sizes)
            ev[k][2].record(stream)
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t_wall0
        sampler.end()
        clocks = sampler.stop()
        res = {"launches": ctx.launches - launches0, "clocks": clocks, "t_wall": t_wall, "sizes": sizes, "out_bytes": out_bytes,
               "payload_bytes": payload_bytes, "prof": ctx.profile_read() if profile else {},
               "tc": sum(ev[k][0].elapsed_time(ev[k][1]) for k in range(steps)) / 1e3,
               "td": sum(ev[k][1].elapsed_time(ev[k][2]) for k in range(steps)) / 1e3,
               "t_total": ev[0][0].elapsed_time(ev[-1][2]) / 1e3}
        if profile:
            ctx.profile(False)
        # lossless round trip of the whole workload, checked on the device outside the timed region (the bit-exactness of
        # the container against the oracle is the parity tests' job: tests/test_gpu_variants.py covers every kernel variant
        # and both container modes on reads drawn by this same generator)
        ok = bool(torch.equal(dec_a[:S], acids_d[:S]) and torch.equal(dec_q[:S], quals_d[:S]))
        if os.environ.get("IDN_BENCH_NOVERIFY"):  # kernel ablation experiments (tools/var_sweep.sh) produce wrong symbols on purpose
            ok = False
        else:
            check_decode_status()
        if not ok and not os.environ.get("IDN_BENCH_NOVERIFY"):
            raise SystemExit(f"round trip mismatch in {mode_name} mode ({name}): the decoded symbols differ from the input")
        res["verified"] = ok
        return res

    main_mode = (args.mode if main else "") or w["mode"]
    other_mode = "native" if main_mode == "compat" else "compat"
    other = None
    if main and not args.no_other_mode and world == 1:  # a short look at the other container format (ratio delta, throughput)
        other = measure(other_mode, 2, 3, False)
    elif not main and world == 1 and main_mode == "native" and not args.no_other_mode:
        other = measure(other_mode, 1, 3, False)  # the ratio delta against the compat output on the same input (north_star)
    m = measure(main_mode, steps, warmup, True)
    if main and args.dump_outputs and rank == 0:  # before the legs below reuse the device buffers
        dump_outputs(Path(args.dump_outputs), chunks, out_d, dec_a, dec_q, S)

    fastq = None
    e2e_file = None
    if main and not args.no_fastq and rank == 0:  # row f1, timed separately: FASTQ text <-> symbols on the device
        fastq = fastq_leg(args, w, capi, torch, ctx, sp, stream, acids_d, quals_d, read_off_h, min(n_reads, 4_000_000))
        if not args.no_e2e:
            e2e_file = e2e_file_leg(args, w, env, acids_d, quals_d, read_off_h, min(n_reads, args.e2e_file_reads))

    extra = after(chunks, out_d, m) if after is not None else None
    e2e = None
    if not args.no_e2e and not no_e2e:  # the host-pointer C-ABI calls on pinned host buffers
        del dec_a, dec_q  # the e2e leg decodes into host buffers; give the device memory back first (torch caches it otherwise,
        torch.cuda.empty_cache()  # and the other contexts of the e2e leg allocate with cudaMalloc)
        e2e = run_e2e(args, w, env, model_names, chunks, acids_d, quals_d, read_off_h, block_first_h, m["sizes"], fq, MODES[main_mode],
                      steps=(args.e2e_steps if main else 2), budget_bytes=(None if main else args.extra_e2e_gb * 1e9))

    rec = {"name": name, "w": w, "mode": main_mode, "n_reads": n_reads, "S": S, "fq": fq, "n_blocks": n_blocks, "chunks": len(chunks),
           "model_names": model_names, "select": select, "m": m, "other": other, "other_mode": other_mode, "e2e": e2e, "fastq": fastq,
           "e2e_file": e2e_file,
           "note": note, "steps": steps, "warmup": warmup, "extra": extra}
    del acids_d, quals_d, out_d, chunks
    torch.cuda.empty_cache()
    return rec


def reduce_record(env, rec):
    """max over ranks of the timed regions; fills the rates of one workload record"""
    m, e2e = rec["m"], rec["e2e"]
    t = [m["t_total"], m["tc"], m["td"], e2e["_t"] if e2e else 0.0]
    if env.dist is not None:
        tt = env.torch.tensor(t, dtype=env.torch.float64, device=env.dev)
        env.dist.all_reduce(tt, op=env.dist.ReduceOp.MAX)
        t = [float(x) for x in tt]
    rec["t_max"], rec["tc_max"], rec["td_max"] = t[0], t[1], t[2]
    if e2e:
        e2e["_t"] = t[3]
    world, fq, steps = env.world, rec["fq"], rec["steps"]
    rec["value"] = 2 * fq * steps * world / rec["t_max"] / 1e9
    rec["compress_GBps"] = fq * steps * world / rec["tc_max"] / 1e9
    rec["decompress_GBps"] = fq * steps * world / rec["td_max"] / 1e9


def roofline_of(rec):
    """roofline of the dominant kernel (by device time inside the timed region) of one workload record"""
    m, S, steps = rec["m"], rec["S"], rec["steps"]
    prof, payload_bytes, out_bytes = m["prof"], m["payload_bytes"], m["out_bytes"]
    peak, peak_src = measured_peak_gbs()
    ksum = sum(ms for _, ms in prof.values()) or 1.0
    dname, (dn, dms) = max(prof.items(), key=lambda kv: kv[1][1])
    # algorithmic bytes per launch (DESIGN.md "Kernels"): encode reads 2 B/symbol and writes the rANS payloads;
    # decode reads the container chunk and writes 2 B/symbol; score reads 2 B/symbol per launch
    per_chunk = rec["chunks"]
    alg = {"encode": (2 * S + payload_bytes) / per_chunk, "decode": (2 * S + out_bytes) / per_chunk,
           "encode_lane": (2 * S + payload_bytes) / per_chunk, "decode_lane": (2 * S + out_bytes) / per_chunk,
           "score": 2 * S / per_chunk, "assemble": 2 * payload_bytes / per_chunk, "crc_read": 2 * S / per_chunk}.get(dname, 2 * S / per_chunk)
    achieved = alg / (dms / dn / 1e3) / 1e9
    traffic = None
    tpath = ROOT / "profiles" / "traffic.json"
    if tpath.exists():
        try:  # measured DRAM bytes per symbol of that kernel (one ncu --set full capture), scaled to this launch size
            traffic = json.loads(tpath.read_text())[dname]["bytes_per_symbol"] * S / per_chunk
        except Exception:
            traffic = None
    return {"bound": "hbm", "kernel": dname + "_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg, "launches_per_step": dn / steps,
            "avg_launch_ms": dms / dn, "share_of_step": dms / ksum,
            "whole_path": {"compress_GBps_alg": (2 * S + out_bytes) * steps / m["tc"] / 1e9,
                           "decompress_GBps_alg": (2 * S + out_bytes) * steps / m["td"] / 1e9},
            "kernels_ms_per_step": {k: v[1] / steps for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}}


def e2e_record(env, rec):
    e2e = rec["e2e"]
    if not e2e:
        return None
    world, fq = env.world, rec["fq"]
    return {"value": 2 * fq * e2e["steps"] * world / e2e["_t"] / 1e9, "unit": "GB/s", "h2d_bytes_per_step": e2e["h2d"],
            "d2h_bytes_per_step": e2e["d2h"], "steps": e2e["steps"], "host_threads": e2e["threads"], "blocks_per_call": e2e["chunk_blocks"],
            "pipeline_blocks": e2e["pipe_blocks"],
            "compress_GBps": e2e["cGBps"] * world, "decompress_GBps": e2e["dGBps"] * world,
            "per_direction_note": "rank 0's own phase times x n_gpus", "sample": e2e["sample"]}


def sub_record(env, rec):
    """what the default run reports for each of the north-star workloads besides the headline one"""
    m, w = rec["m"], rec["w"]
    rf = roofline_of(rec)
    out = {"workload": w["desc"], "mode": rec["mode"], "reads_per_gpu": rec["n_reads"], "fastq_bytes_per_gpu": rec["fq"],
           "blocks_per_gpu": rec["n_blocks"], "models": rec["model_names"], "steps": rec["steps"], "warmup": rec["warmup"],
           "value": rec["value"], "unit": "GB/s", "compress_GBps": rec["compress_GBps"], "decompress_GBps": rec["decompress_GBps"],
           "ms_per_step": rec["t_max"] / rec["steps"] * 1e3, "container_bytes_per_read": m["out_bytes"] / rec["n_reads"],
           "bits_per_base": 8 * m["payload_bytes"] / rec["S"], "verified_round_trip": m["verified"], "gpu_launches": m["launches"],
           "clocks": m["clocks"],
           "roofline": {k: rf[k] for k in ("kernel", "achieved", "peak", "frac", "algorithmic_bytes_per_launch", "avg_launch_ms",
                                           "share_of_step", "kernels_ms_per_step")},
           "e2e": e2e_record(env, rec)}
    if rec["other"]:
        o = rec["other"]
        out["ratio_delta_vs_" + rec["other_mode"]] = {"container_bytes_per_read": o["out_bytes"] / rec["n_reads"],
                                                      "size_vs_" + rec["other_mode"]: m["out_bytes"] / o["out_bytes"],
                                                      "verified_round_trip": o["verified"]}
    if rec["note"]:
        out["note"] = rec["note"]
    return out


def run_strong(env, args):
    """ONE file shared by all ranks (strong scaling): the NovaSeq-shaped 50 GB workload of BASELINE.json configs[2] is cut into
    contiguous block ranges, one per GPU (blocks are independent, compressor_block.rs:61-62); every rank compresses and
    decompresses its range with its inputs resident in HBM; the ranks then exchange their container sizes (the offset
    prefix sum -- the only communication of the path) and each writes its range at its offset into one file in /dev/shm,
    which rank 0 walks from the first block header to the last.  The N-GPU == 1-GPU byte identity of such a concatenation is
    tests/test_gpu_pipeline.py's business; here it is timed."""
    import mmap
    torch, dist, rank, world = env.torch, env.dist, env.rank, env.world
    w = dict(WORKLOADS["novaseq150_native"])
    total_reads = w["reads"]
    per_block = max(1, BLOCK_SYMBOLS // w["read_len"][0])
    total_blocks = -(-total_reads // per_block)
    b0, b1 = total_blocks * rank // world, total_blocks * (rank + 1) // world
    r0, r1 = min(total_reads, b0 * per_block), min(total_reads, b1 * per_block)
    path = f"/dev/shm/idn_strong_{os.environ.get('MASTER_PORT', '0')}.idn"
    res = {}

    def concat(chunks, out_d, m):
        """sizes -> offsets -> every rank writes its bytes at its offset (timed: D2H + the write into the shared file)"""
        mine = sum(m["sizes"].values())
        sizes = torch.zeros(world, dtype=torch.int64, device=env.dev)
        sizes[rank] = mine
        dist.all_reduce(sizes)
        sizes = sizes.cpu().numpy()
        off = int(sizes[:rank].sum())
        total = int(sizes.sum())
        if rank == 0:
            with open(path, "wb") as f:
                f.truncate(total)
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with open(path, "r+b") as f:
            mm = mmap.mmap(f.fileno(), 0)
            dst = np.frombuffer(mm, dtype=np.uint8)
            pos = off
            for c in chunks:
                n = m["sizes"][id(c)]
                t = torch.from_numpy(dst[pos:pos + n])
                t.copy_(out_d[c.out_base:c.out_base + n])  # D2H straight into the shared mapping
                pos += n
            torch.cuda.synchronize()
            del dst, t
            mm.close()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=env.dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        res["concat_s"] = float(tt[0])
        res["container_bytes"] = total
        dist.barrier()
        if rank == 0:  # the concatenation is one valid block sequence
            buf = np.memmap(path, dtype=np.uint8, mode="r")
            pos, nb = 0, 0
            while pos < total:
                ln = int.from_bytes(bytes(buf[pos:pos + 4]), "big")
                pos += 8 + ln
                nb += 1
            res["blocks_walked"] = nb
            res["walk_ok"] = bool(pos == total and nb == total_blocks)
            del buf
            os.unlink(path)
        return None

    rec = run_workload(env, args, "novaseq150_native", w, steps=args.extra_steps, warmup=3, main=False, shard=(r0, r1 - r0), no_e2e=True,
                       after=concat)
    # one file: the time of the slowest rank bounds the file
    t = torch.tensor([rec["m"]["t_total"], rec["m"]["tc"], rec["m"]["td"]], dtype=torch.float64, device=env.dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    fq_total = fastq_bytes(w, total_reads, total_reads * w["read_len"][0])
    steps = rec["steps"]
    out = {"workload": w["desc"] + ": ONE file, contiguous block ranges over the GPUs", "scaling": "strong", "reads_total": total_reads,
           "fastq_bytes_total": fq_total, "blocks_total": total_blocks, "blocks_of_rank0": b1 - b0 if rank == 0 else None,
           "value": 2 * fq_total * steps / float(t[0]) / 1e9, "compress_GBps": fq_total * steps / float(t[1]) / 1e9,
           "decompress_GBps": fq_total * steps / float(t[2]) / 1e9, "unit": "GB/s", "steps": steps,
           "concat_ms": res.get("concat_s", 0.0) * 1e3, "container_bytes": res.get("container_bytes"),
           "compress_plus_concat_GBps": fq_total / (float(t[1]) / steps + res.get("concat_s", 0.0)) / 1e9,
           "blocks_walked": res.get("blocks_walked"), "concatenation_is_one_block_sequence": res.get("walk_ok"),
           "verified_round_trip": rec["m"]["verified"],
           "note": "device-resident per-rank timing, max over ranks; concat = D2H of every rank's range into one /dev/shm file at its "
                   "prefix-sum offset (max over ranks), no collective on the data path"}
    return out


def run_gpu(args, w: dict):
    env = setup_gpu()
    rank, world = env.rank, env.world
    rec = run_workload(env, args, args.workload, w, steps=args.steps, warmup=args.warmup, main=True)
    reduce_record(env, rec)
    extras = {}
    if args.extra_workloads and not (args.acid or args.q or args.reads):
        for xname in EXTRA_WORKLOADS:
            if xname == args.workload or WORKLOADS[xname] is w:
                continue
            x = run_workload(env, args, xname, dict(WORKLOADS[xname]), steps=args.extra_steps, warmup=3, main=False)
            reduce_record(env, x)
            extras[xname] = x
    few = None
    if "pacbio_native" in extras:
        # the point of cutting long reads into lanes: throughput no longer needs ~150 k reads in flight.  10 000 long reads
        # (one thread per read: 7 % of the GPU's thread slots) in both container modes
        few = {}
        for xname in ("pacbio", "pacbio_native"):
            x = run_workload(env, args, xname, dict(WORKLOADS[xname]), steps=3, warmup=3, main=False, shard=(rank * 10_000, 10_000), no_e2e=True)
            reduce_record(env, x)
            few[WORKLOADS[xname]["mode"]] = {"reads_per_gpu": 10_000, "value": x["value"], "compress_GBps": x["compress_GBps"],
                                              "decompress_GBps": x["decompress_GBps"], "verified_round_trip": x["m"]["verified"]}
    strong = None
    if world > 1 and args.extra_workloads and not (args.acid or args.q or args.reads):
        strong = run_strong(env, args)
    if rank == 0:
        m = rec["m"]
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline(args, w)
        S, n_reads, fq = rec["S"], rec["n_reads"], rec["fq"]
        line = {
            "metric": "fastq_compress_decompress_GBps", "value": rec["value"], "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": rec["t_max"] / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic (model-driven sampler, SURVEY.md 8d)",
            "config": {"workload": w["desc"], "name": args.workload, "mode": rec["mode"], "acid_model": w["acid"], "q_model": w["q"],
                       "reads_per_gpu": n_reads, "symbols_per_gpu": S, "fastq_bytes_per_gpu": fq, "blocks_per_gpu": rec["n_blocks"],
                       "block_symbols": BLOCK_SYMBOLS, "chunk_blocks": args.chunk_blocks,
                       "names": "not stored (--no-identifiers protocol, util/benchmark.py:161-179); their bytes count as FASTQ input: the "
                                f"kernels touch the {2 * S / 1e9:.1f} GB of symbols of the {fq / 1e9:.1f} GB of FASTQ text (both arms alike)",
                       "l2": f"inputs {2 * S / 1e9:.1f} GB >> 126 MB L2, no flush needed",
                       "model_selection": ("explicit pair (1 acid + 1 q-score model), quality 7 semantics" if rec["select"] <= 1 else
                                           "per-read greedy selection among the models quality 7 retains from models/"),
                       "models": rec["model_names"],
                       "parity": "round trip verified here; bit-exactness against the oracle: tests/test_gpu_variants.py, tests/test_gpu_parity.py"},
            "compress_GBps": rec["compress_GBps"], "decompress_GBps": rec["decompress_GBps"],
            "container_bytes_per_read": m["out_bytes"] / n_reads, "bits_per_base": 8 * m["payload_bytes"] / S,
            "verified_round_trip": m["verified"], "gpu_launches": m["launches"], "clocks": m["clocks"], "roofline": roofline_of(rec),
            "wall_s_timed": m["t_wall"],
        }
        e = e2e_record(env, rec)
        if e:
            line["e2e"] = e
        if cpu:
            line["cpu_baseline"] = cpu
        if rec["fastq"]:
            line["fastq_text"] = rec["fastq"]
        if rec["e2e_file"]:
            line["e2e_file"] = rec["e2e_file"]
        if rec["other"]:
            o = rec["other"]
            line["other_mode"] = {"mode": rec["other_mode"], "compress_GBps": fq * 2 / o["tc"] / 1e9, "decompress_GBps": fq * 2 / o["td"] / 1e9,
                                  "container_bytes_per_read": o["out_bytes"] / n_reads, "verified_round_trip": o["verified"],
                                  "size_vs_main_mode": o["out_bytes"] / m["out_bytes"], "steps": 2, "n_gpus": 1,
                                  "note": "this rank only, device-resident, 2 timed steps"}
        if extras:
            line["workloads"] = {k: sub_record(env, x) for k, x in extras.items()}
            if few:
                line["workloads"]["pacbio_native"]["with_10k_reads_in_flight"] = few
        if strong:
            line["strong_scaling"] = strong
        print(json.dumps(line))
    if env.dist is not None:
        env.dist.barrier()
        env.dist.destroy_process_group()
    env.ctx.close()


def fastq_leg(args, w, capi, torch, ctx, sp, stream, acids_d, quals_d, read_off_h, n):
    """FASTQ text of the first n reads is produced on the device (format), parsed back (parse) and compared."""
    L = ctx.L
    dev = acids_d.device
    S = int(read_off_h[n])
    ro_d = torch.from_numpy(read_off_h[:n + 1].view(np.int64)).to(dev)
    # fixed-width synthetic titles "r000000000123 1:N:0"
    idx = torch.arange(n, dtype=torch.int64, device=dev)
    digits = torch.stack([(idx // 10 ** k) % 10 for k in range(11, -1, -1)], dim=1).to(torch.uint8) + 48
    tail = torch.tensor(list(b" 1:N:0"), dtype=torch.uint8, device=dev).expand(n, -1)
    head = torch.full((n, 1), ord("r"), dtype=torch.uint8, device=dev)
    names_d = torch.cat([head, digits, tail], dim=1).contiguous().view(-1)
    nlen = 1 + 12 + 6
    no_d = (torch.arange(n + 1, dtype=torch.int64, device=dev) * nlen).contiguous()
    b = capi.Batch()
    b.n_reads, b.n_symbols, b.n_blocks = n, S, 0
    b.acids, b.quals, b.read_off = acids_d.data_ptr(), quals_d.data_ptr(), ro_d.data_ptr()
    b.names, b.name_off = names_d.data_ptr(), no_d.data_ptr()
    cap = 2 * S + n * (6 + nlen) + 64
    text_d = torch.empty(cap, dtype=torch.uint8, device=dev)
    n_out = torch.zeros(1, dtype=torch.int64, device=dev)
    info = capi.FastqInfo()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    for it in range(3):  # two warm-ups, the third pass is timed
        ev[0].record(stream)
        ctx.check(L.idn_gpu_fastq_format_dev(ctx.h, C.byref(b), 0, text_d.data_ptr(), cap, n_out.data_ptr(), sp))
        ev[1].record(stream)
        torch.cuda.synchronize()
        nbytes = int(n_out.item())
        ev[2].record(stream)
        ctx.check(L.idn_gpu_fastq_parse_dev(ctx.h, text_d.data_ptr(), nbytes, C.byref(info), sp))
        ev[3].record(stream)
        torch.cuda.synchronize()
    # compare on the host (outside the timed passes)
    chk_a = np.zeros(max(S, 1), dtype=np.uint8)
    chk_q = np.zeros(max(S, 1), dtype=np.uint8)
    ctx.check(L.idn_gpu_fastq_fetch(ctx.h, chk_a.ctypes.data, chk_q.ctypes.data, None, None, None))
    ok = bool(info.n_reads == n and info.n_symbols == S and np.array_equal(chk_a[:S], acids_d[:S].cpu().numpy()) and
              np.array_equal(chk_q[:S], quals_d[:S].cpu().numpy()))
    if not ok:
        raise SystemExit("FASTQ text round trip mismatch")
    return {"sample": f"first {n} reads, {nbytes / 1e9:.2f} GB of FASTQ text, device-resident, third of three passes",
            "format_GBps": nbytes / (ev[0].elapsed_time(ev[1]) / 1e3) / 1e9, "parse_GBps": nbytes / (ev[2].elapsed_time(ev[3]) / 1e3) / 1e9,
            "verified_round_trip": ok}


def e2e_file_leg(args, w, env, acids_d, quals_d, read_off_h, n):
    """FASTQ TEXT in host memory -> .idn bytes in host memory -> FASTQ text in host memory, through the host mirror of the
    reference API (IdnCompressor::add_fastq_text / IdnDecompressor::next_fastq_text, csrc/host/idn.cpp): the text is uploaded
    once, split into records and blocks and compressed on the device; the identifiers go through the host's Deflate.  Timed
    with and without identifiers (north_star: the name codec stays on the host and is timed separately), on the first n
    reads of the workload with synthetic titles.  Wall clock of the calls, everything included."""
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    torch, capi, host, ctx = env.torch, env.capi, env.host, env.ctx
    L, dev, sp = ctx.L, env.dev, env.sp
    S = int(read_off_h[n])
    ro_d = torch.from_numpy(read_off_h[:n + 1].view(np.int64)).to(dev)
    idx = torch.arange(n, dtype=torch.int64, device=dev)
    digits = torch.stack([(idx // 10 ** k) % 10 for k in range(11, -1, -1)], dim=1).to(torch.uint8) + 48
    tail = torch.tensor(list(b" 1:N:0"), dtype=torch.uint8, device=dev).expand(n, -1)
    head = torch.full((n, 1), ord("r"), dtype=torch.uint8, device=dev)
    names_d = torch.cat([head, digits, tail], dim=1).contiguous().view(-1)
    nlen = 1 + 12 + 6
    no_d = (torch.arange(n + 1, dtype=torch.int64, device=dev) * nlen).contiguous()
    b = capi.Batch()
    b.n_reads, b.n_symbols, b.n_blocks = n, S, 0
    b.acids, b.quals, b.read_off = acids_d.data_ptr(), quals_d.data_ptr(), ro_d.data_ptr()
    b.names, b.name_off = names_d.data_ptr(), no_d.data_ptr()
    cap = 2 * S + n * (6 + nlen) + 64
    text_d = torch.empty(cap, dtype=torch.uint8, device=dev)
    n_out = torch.zeros(1, dtype=torch.int64, device=dev)
    ctx.check(L.idn_gpu_fastq_format_dev(ctx.h, C.byref(b), 0, text_d.data_ptr(), cap, n_out.data_ptr(), sp))
    torch.cuda.synchronize()
    nbytes = int(n_out.item())
    text_h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    text_h.copy_(text_d[:nbytes])
    torch.cuda.synchronize()
    text_np = text_h.numpy()
    names_h = names_d.cpu().numpy()
    del text_d, names_d, digits
    torch.cuda.empty_cache()
    models = [host.Model.load(MODELS / (w["acid"] + ".msgpack")), host.Model.load(MODELS / (w["q"] + ".msgpack"))]
    cores = os.cpu_count() or 1
    out = {"sample": f"first {n} reads as {nbytes / 1e9:.2f} GB of FASTQ text (titles of {nlen} bytes), page-locked host memory in, host memory out",
           "host_threads_for_identifiers": cores}
    idn_h = torch.empty(nbytes // 2 + (64 << 20), dtype=torch.uint8, pin_memory=True).numpy()  # the ".idn file"
    back_h = torch.empty(nbytes + 64, dtype=torch.uint8, pin_memory=True).numpy()               # the text "file" written back
    devs = [env.local, env.local]  # two contexts on the device: one batch's copies overlap the other's kernels
    out["contexts_on_the_device"] = len(devs)
    for names in (False, True):
        best = None
        for it in range(4):  # the last pass is the timed one: the library keeps device contexts and page-locked buffers
            # between objects (sized by the passes before), as a process that compresses more than one file would find them
            c = host.IdnCompressor(models, include_identifiers=names, thread_num=cores, devices=devs,
                                   text_chunk_bytes=args.text_chunk_mb << 20, batch_blocks=args.file_batch_blocks)
            c.set_output(idn_h)
            t0 = time.perf_counter()
            c.add_fastq_text(text_np)
            c.finish(copy=False)
            t1 = time.perf_counter()
            idn = c.output_view()
            n_idn = int(idn.size)
            # (1) streaming: the text of each batch of blocks is handed out where the device wrote it (what a writer passes to write())
            t2 = time.perf_counter()
            rd = host.FastqTextReader(models, idn, devices=devs, thread_num=cores, batch_blocks=args.file_batch_blocks)
            t2a = time.perf_counter()
            got = 0
            for piece in rd:
                got += piece.size
            t2b = time.perf_counter()
            rd.close()
            t3 = time.perf_counter()
            if os.environ.get("IDN_HOST_TRACE"):
                print(f"[bench e2e_file] pass {it} names {names}: compress {t1 - t0:.3f} s; reader open {t2a - t2:.3f} pieces {t2b - t2a:.3f} close {t3 - t2b:.3f} s",
                      file=sys.stderr, flush=True)
            # (2) the same into one contiguous caller buffer (one more host copy)
            n_back = host.decompress_text_into(models, idn, back_h, device=env.local, thread_num=cores, batch_blocks=args.file_batch_blocks)
            t4 = time.perf_counter()
            back = back_h[:n_back]
            if names:
                ok = got == nbytes and n_back == nbytes and bool(np.array_equal(back, text_np))
            else:  # empty titles: the symbol lines only
                ok = got == nbytes - n * nlen and n_back == got
            c.close()
            best = (t1 - t0, t3 - t2, t4 - t3, n_idn, ok)
        tc, td, td2, n_idn, ok = best
        if not ok:
            raise SystemExit("e2e_file: the text that came back differs from the text that went in")
        out["with_identifiers" if names else "no_identifiers"] = {
            "compress_GBps": nbytes / tc / 1e9, "decompress_GBps": nbytes / td / 1e9, "value": 2 * nbytes / (tc + td) / 1e9,
            "decompress_into_one_buffer_GBps": nbytes / td2 / 1e9, "container_bytes": n_idn, "verified_round_trip": ok}
    host.release_cached()  # the contexts and page-locked buffers the host mirror keeps between objects
    del idn_h, back_h
    # the identifiers codec alone, as the host mirror runs it: raw Deflate level 6 per block on `cores` threads
    per_block = max(1, BLOCK_SYMBOLS // int(read_off_h[1] - read_off_h[0])) if n else 1
    blocks = [b"\n".join(bytes(names_h[r * nlen:(r + 1) * nlen]) for r in range(b0, min(n, b0 + per_block))) for b0 in range(0, min(n, 16 * per_block), per_block)]
    raw = sum(len(x) for x in blocks)

    def deflate(x):
        z = zlib.compressobj(6, zlib.DEFLATED, -15)
        return z.compress(x) + z.flush()
    with ThreadPoolExecutor(cores) as ex:
        t0 = time.perf_counter()
        zs = list(ex.map(deflate, blocks))
        t1 = time.perf_counter()
        back = list(ex.map(lambda z: zlib.decompress(z, -15), zs))
        t2 = time.perf_counter()
    assert back == blocks
    out["identifiers_codec_alone"] = {"names_deflate_GBps": raw / (t1 - t0) / 1e9, "names_inflate_GBps": raw / (t2 - t1) / 1e9,
                                      "threads": cores, "sample_bytes": raw, "ratio": sum(len(z) for z in zs) / max(raw, 1),
                                      "note": "zlib level 6 raw Deflate per block (the reference uses flate2/miniz_oxide at its default level)"}
    return out


def cpu_baseline(args, w: dict) -> dict:
    cores = os.cpu_count() or 1
    n_blocks = args.cpu_blocks or max(8, min(2 * cores, 256))
    O, models, reads = cpu_sample(w, n_blocks, cores)
    fq = fastq_bytes(w, reads.n_reads, int(reads.read_off[-1]))
    cpu_step(O, models, reads, cores)  # warm-up
    tc, td, _ = cpu_step(O, models, reads, cores)
    return {"value": 2 * fq / (tc + td) / 1e9, "unit": "GB/s", "cores": cores, "kind": "port",
            "sample": f"first {reads.n_reads} reads ({n_blocks} blocks, {fq / 1e6:.0f} MB FASTQ) of the workload, one timed pass after one warm-up",
            "compress_GBps": fq / tc / 1e9, "decompress_GBps": fq / td / 1e9,
            "note": "reference-algorithm CPU restatement (oracle/), one worker thread per block like idn/thread_pool.rs"}


def run_e2e(args, w, env, model_names, chunks, acids_d, quals_d, read_off_h, block_first_h, sizes, fq_total, mode, *, steps, budget_bytes):
    """Same step through idn_gpu_compress_blocks / idn_gpu_decompress_blocks with HOST buffers."""
    import psutil
    torch, capi, host, local, dist = env.torch, env.capi, env.host, env.local, env.dist
    S = int(read_off_h[-1])
    total_out = sum(sizes.values())
    # A host-pointer call pipelines itself (csrc/idn_pipeline.inc: sub-chunks of blocks on an upload, a compute and a download
    # stream), so ONE context on ONE host thread gets a whole direction in one call; --e2e-threads / --e2e-chunk-blocks
    # reproduce round 1's several-contexts-in-flight arrangement for comparison.
    n_blocks_all = len(block_first_h) - 1
    reads_per_block = max(1, (len(read_off_h) - 1) // max(n_blocks_all, 1))
    # a sub-chunk should carry enough reads to fill the GPU (one thread per read: ~150 k in flight): blocks of long reads
    # hold a few hundred reads each, so those workloads pipeline in larger sub-chunks
    per_call = E2E_READS_PER_CALL_COMPAT if mode == capi.MODE_COMPAT else E2E_READS_PER_CALL
    pipe_blocks = args.e2e_pipe_blocks or max(32, min(256, -(-per_call // reads_per_block)))
    # pinned inputs, pinned container, pinned decoded output: 4 * S + 2 * container bytes of page-locked host memory.  Budget
    # of this rank: half of what is available, shared by the ranks of the box (or the caller's limit); a workload that
    # needs more is sampled from its front and the rate scaled
    need = 4 * S + total_out * 2
    budget = 0.5 * psutil.virtual_memory().available / max(1, int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1"))))
    if budget_bytes:
        budget = min(budget, budget_bytes)
    use_blocks = n_blocks_all
    if need > budget:
        use_blocks = max(min(n_blocks_all, 4 * pipe_blocks), int(n_blocks_all * budget / need))
    chunk_blocks = args.e2e_chunk_blocks
    if chunk_blocks <= 0:  # automatic: all blocks of a thread in one call
        chunk_blocks = max(1, -(-use_blocks // max(1, args.e2e_threads)))
    e2e_chunks = []
    for b0 in range(0, use_blocks, chunk_blocks):
        c = Chunk()
        c.b0, c.b1 = b0, min(use_blocks, b0 + chunk_blocks)
        c.r0, c.r1 = int(block_first_h[c.b0]), int(block_first_h[c.b1])
        c.s0, c.s1 = int(read_off_h[c.r0]), int(read_off_h[c.r1])
        c.n_reads, c.n_syms, c.n_blocks = c.r1 - c.r0, c.s1 - c.s0, c.b1 - c.b0
        e2e_chunks.append(c)
    per_sym = total_out / max(S, 1)
    sizes = {id(c): int(per_sym * c.n_syms * 1.15) + 64 * c.n_blocks + 4096 for c in e2e_chunks}  # container capacity per call
    chunks = e2e_chunks
    n_threads = max(1, min(args.e2e_threads, len(chunks)))
    use = chunks
    s_end = use[-1].s1
    r_end = use[-1].r1
    acids_h = torch.empty(s_end, dtype=torch.uint8, pin_memory=True)
    quals_h = torch.empty(s_end, dtype=torch.uint8, pin_memory=True)
    acids_h.copy_(acids_d[:s_end])
    quals_h.copy_(quals_d[:s_end])
    torch.cuda.synchronize()
    a_np, q_np = acids_h.numpy(), quals_h.numpy()
    stride = (max(sizes[id(c)] for c in use) * 21 // 20 + 4096) // 256 * 256
    cont_h = torch.empty(stride * len(use), dtype=torch.uint8, pin_memory=True)
    cont_np = cont_h.numpy()
    da_h = torch.empty(s_end, dtype=torch.uint8, pin_memory=True)
    dq_h = torch.empty(s_end, dtype=torch.uint8, pin_memory=True)
    da_np, dq_np = da_h.numpy(), dq_h.numpy()
    ctxs = []
    for _ in range(n_threads):
        cx = capi.Context(local)
        cx.set_pipeline_blocks(pipe_blocks)
        ctxs.append((cx, np.asarray([host.Model.load(MODELS / (st + ".msgpack")).upload(cx) for st in model_names], dtype=np.int32)))
    n_models = len(model_names)

    def pinned(n, dtype):
        """every buffer the C-ABI calls copy from / to is page-locked (a pageable copy is staged and synchronous)"""
        t = torch.empty(max(int(n), 1), dtype=dtype, pin_memory=True)
        return t, t.numpy()

    per_chunk = []
    for i, c in enumerate(use):
        ro_t, ro = pinned(c.n_reads + 1, torch.int64)
        ro[:c.n_reads + 1] = (read_off_h[c.r0:c.r1 + 1] - read_off_h[c.r0]).view(np.int64)
        bf_t, bf = pinned(c.n_blocks + 1, torch.int32)
        bf[:c.n_blocks + 1] = (block_first_h[c.b0:c.b1 + 1] - block_first_h[c.b0]).astype(np.int32)
        boff_t, boff = pinned(c.n_blocks + 1, torch.int64)
        crc_t, crc = pinned(c.n_blocks, torch.int32)
        doff_t, doff = pinned(c.n_blocks + 1, torch.int64)
        dlen_t, dlen = pinned(c.n_blocks, torch.int32)
        roo_t, roo = pinned(c.n_reads + 1, torch.int64)
        b = capi.Batch()
        b.n_reads, b.n_symbols, b.n_blocks = c.n_reads, c.n_syms, c.n_blocks
        b.acids, b.quals = a_np.ctypes.data + c.s0, q_np.ctypes.data + c.s0
        b.read_off, b.block_first_read = ro.ctypes.data, bf.ctypes.data
        per_chunk.append(dict(batch=b, keep=(ro_t, bf_t, boff_t, crc_t, doff_t, dlen_t, roo_t), block_off=boff.view(np.uint64),
                              crc=crc.view(np.uint32), doff=doff.view(np.uint64), dlen=dlen.view(np.uint32),
                              stats=capi.CompressStats(), ro_out=roo.view(np.uint64), bad=C.c_int32(-1)))
    errors = []

    def worker(t, phase):
        cx, hd = ctxs[t]
        L = cx.L
        try:
            for i in range(t, len(use), n_threads):
                c, pc = use[i], per_chunk[i]
                base = cont_np.ctypes.data + i * stride
                if phase == 0:
                    cx.check(L.idn_gpu_compress_blocks(cx.h, C.byref(pc["batch"]), mode, hd.ctypes.data, n_models, 0, None,
                                                       base, stride, pc["block_off"].ctypes.data, pc["crc"].ctypes.data,
                                                       C.byref(pc["stats"])))
                else:
                    bo, doff, dlen = pc["block_off"], pc["doff"], pc["dlen"]
                    nb = c.n_blocks
                    doff[:nb] = bo[:nb] + 8
                    doff[nb] = bo[nb]
                    dlen[:nb] = (bo[1:nb + 1] - bo[:nb] - 8).astype(np.uint32)
                    cx.check(L.idn_gpu_decompress_blocks(cx.h, base, doff.ctypes.data, dlen.ctypes.data, pc["crc"].ctypes.data,
                                                         c.n_blocks, mode, hd.ctypes.data, n_models, None, None,
                                                         da_np.ctypes.data + c.s0, dq_np.ctypes.data + c.s0,
                                                         pc["ro_out"].ctypes.data, c.n_reads, c.n_syms, C.byref(pc["bad"])))
        except Exception as e:  # surfaced after the join
            errors.append(e)

    def phase(p):
        ts = [threading.Thread(target=worker, args=(t, p)) for t in range(n_threads)]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        torch.cuda.synchronize()
        if errors:
            raise errors[0]
        return time.perf_counter() - t0

    steps = max(1, steps)
    for _ in range(2):  # warm-up: sizes the staging buffers of every ctx
        phase(0)
        phase(1)
    if args.e2e_profile:
        for cx, _ in ctxs:
            cx.profile(True)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    tc = td = 0.0
    t0 = time.perf_counter()
    for _ in range(steps):
        tc += phase(0)
        td += phase(1)
    t_all = time.perf_counter() - t0
    if args.e2e_profile:
        agg = {}
        for cx, _ in ctxs:
            for k, (n, ms) in cx.profile_read().items():
                a = agg.setdefault(k, [0, 0.0])
                a[0] += n
                a[1] += ms
            cx.profile(False)
        print("e2e phases (summed over ctx, ms per step):", {k: (v[0] // steps, round(v[1] / steps, 1)) for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])},
              file=sys.stderr)
    ok = np.array_equal(da_np[:s_end], a_np[:s_end]) and np.array_equal(dq_np[:s_end], q_np[:s_end])
    if not ok:
        raise SystemExit("e2e round trip mismatch")
    for cx, _ in ctxs:
        cx.close()
    frac = s_end / S
    fq = fq_total * frac
    cbytes = sum(int(pc["stats"].out_bytes) for pc in per_chunk)
    h2d = 2 * s_end + 8 * (r_end + len(use)) + cbytes
    d2h = cbytes + 2 * s_end + 8 * (r_end + len(use))
    return {"_t": t_all / frac, "steps": steps, "h2d": int(h2d / frac), "d2h": int(d2h / frac), "threads": n_threads, "chunk_blocks": chunk_blocks,
            "pipe_blocks": pipe_blocks,
            "cGBps": fq * steps / tc / 1e9, "dGBps": fq * steps / td / 1e9,
            "sample": "whole workload" if use_blocks == n_blocks_all else
                      f"first {use_blocks} of {n_blocks_all} blocks ({fq / 1e9:.1f} GB of FASTQ; pinned host memory budget), scaled"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="hiseq100", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extra-workloads", dest="extra_workloads", action="store_false",
                    help="skip the sub-records of the other north-star workloads (NovaSeq native, PacBio, per-read selection)")
    ap.add_argument("--extra-steps", type=int, default=5, help="timed steps of each extra workload")
    ap.add_argument("--extra-e2e-gb", type=float, default=6.0, help="pinned host memory of the e2e leg of an extra workload (a sample, scaled)")
    ap.add_argument("--reads", type=int, default=0, help="reads per GPU (default: the workload's)")
    ap.add_argument("--acid", default="", help="acid model (file stem in models/) instead of the workload's")
    ap.add_argument("--q", default="", help="quality score model (file stem in models/) instead of the workload's")
    ap.add_argument("--chunk-blocks", type=int, default=1024, help="blocks per library call of the device-resident leg")
    ap.add_argument("--full-bound", action="store_true", help="size container chunks by idn_gpu_compress_bound")
    ap.add_argument("--cpu-blocks", type=int, default=0, help="blocks in the CPU sample (default 2 per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-fastq", action="store_true", help="skip the FASTQ text parse/format leg (row f1)")
    ap.add_argument("--select", type=int, default=1, help="> 1: per-read selection among the 4 + 4 models quality 7 retains from models/")
    ap.add_argument("--mode", default="", choices=["", "compat", "native"], help="container format (default: the workload's)")
    ap.add_argument("--no-other-mode", action="store_true", help="skip the short run of the other container format")
    ap.add_argument("--lane-symbols", type=int, default=0, help="native mode lane quantum (default: the library's 2048)")
    ap.add_argument("--e2e-threads", type=int, default=1, help="host threads (one ctx each) of the e2e leg")
    ap.add_argument("--e2e-chunk-blocks", type=int, default=0, help="blocks per host-pointer call in the e2e leg (default: all of a thread's blocks in one call)")
    ap.add_argument("--e2e-pipe-blocks", type=int, default=0, help="blocks per sub-chunk of the pipeline inside a call (default: 32, more for long reads)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-file-reads", type=int, default=24_000_000, help="reads of the FASTQ-text-in / text-out leg through the host mirror")
    ap.add_argument("--text-chunk-mb", type=int, default=256, help="FASTQ text per device call of that leg")
    ap.add_argument("--file-batch-blocks", type=int, default=32, help="blocks per batch in the e2e_file decode (and in add_batch)")
    ap.add_argument("--e2e-profile", action="store_true", help="print the host-side phase times of the e2e leg to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed step of the headline workload to DIR/<name>.npy (GPU arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.warmup < 3:
        args.warmup = 3
    w = dict(WORKLOADS[args.workload])
    if args.acid or args.q:
        w["acid"], w["q"] = args.acid or w["acid"], args.q or w["q"]
        w["desc"] += f" [models overridden: {w['acid']} + {w['q']}]"
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_gpu(args, w)


if __name__ == "__main__":
    main()

"""Per-read model selection against the CPU oracle at the shapes where its kernels branch.

With several models per type (quality >= 2 keeps up to 4 + 4; any caller may pass up to 16 + 16) the device scores every
read under every candidate (score_multi_kernel), picks a model per read (switch_kernel, compat format) or per lane
(lane_choose_kernel, native format), buckets the reads / lanes by the chosen (acid, q-score) pair (bucket_count / base /
scatter) and launches the uniform kernel of every pair over its list (encode_list_kernel, decode_list_kernel,
encode_lane_list_kernel, decode_lane_list_kernel; a fixed grid of sm_count x 8 CTAs of 128 threads striding over the
list).  Without buckets (IDN_NO_BUCKETS=1, or a decode with more than 32 models) the run-time-generic kernels run instead.

A wrong choice does not break the round trip -- the decoder follows whatever SwitchModel slices or lane table the encoder
wrote -- it breaks bit-identity with the reference.  So every test here compares bytes with the oracle:

* two plain references, checked against the oracle's own containers on the CPU (no GPU needed): a walker over the
  slices of a compat block that returns the models in force for every read, and a restatement of the greedy chooser;
* 9 + 9 candidates (one pair per compile-time-specialised kernel variant plus the generic salmonella pair) on a batch
  mixed from runs of 1-64 reads of each pair, with one HiSeq run long enough that the list kernels stride over their
  bucket at least twice: choices against the restatement, scores against the oracle, containers byte for byte, decode;
* ties: a twin model that scores like its original on every read, in both orders, at block sizes around the warp size;
* limits: 16 + 16 candidates (1024 pairs on the decode side), a 17th refused, a 17 + 17 container decoded through the
  generic fallback, and all of the above again with IDN_NO_BUCKETS=1;
* the host mirror with all 22 bundled models at the shape of bench.py's hiseq100_select4 workload.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import MODELS, ROOT
from gpu_util import PAIRS, SPEC_NAMES, blocks_of, parse_compat_block, synth_on_device, synthetic_model, toy_reads, upload

COMPAT, NATIVE = 1, 2
BLOCK = 4 * 1024 * 1024
SWITCH_PENALTY = 2           # bytes charged to a model that is not the active one (model_chooser.rs:175-186)
LIST_CTAS_PER_SM = 8         # IDN_ENC_MINB / IDN_DEC_MINB / IDN_LANE_MINB: grid of the list kernels
LIST_THREADS = 128
THREADS = os.cpu_count() or 8

# one pair per specialised kernel variant (SP0..SP7) plus the generic one (salmonella: hashed 2^27-spec q-score model)
SELECT_PAIRS = ["hiseq2000", "novaseq_human", "sequel2", "novaseq_cat", "hiseq2500_cat", "iseq100", "hiseq2500_e_coli",
                "hiseq2500_pear", "hiseq2500_salmonella"]


# ---- plain references (no GPU) ---------------------------------------------------------------------------------------
def _u32(buf, pos):
    return int.from_bytes(buf[pos:pos + 4], "big")


def split_container(idn: bytes):
    """IdnHeader, metadata and blocks {u32be length, u32be crc32, slices} up to the empty terminator block
    (writer_idn.rs:25-59) -> (version, model identifiers, [(slices, crc)])"""
    assert idn[:8] == b"IDENCOMP" and idn[9:11] == b"\x01\x00"
    n = idn[11]
    ids = [idn[12 + 32 * i:12 + 32 * (i + 1)] for i in range(n)]
    pos, blocks = 12 + 32 * n, []
    while True:
        ln, crc = _u32(idn, pos), _u32(idn, pos + 4)
        pos += 8
        if ln == 0:
            break
        blocks.append((idn[pos:pos + ln], crc))
        pos += ln
    assert pos == len(idn)
    return idn[8], ids, blocks


def native_lane_models(data: bytes):
    """The lane model table of the NativeLanes slice of one version-2 block (idn_native.cuh header) -> [n_lanes, 2]
    container model indices (acid, q-score)"""
    pos = 0
    if data[0] == 0:  # Identifiers slice
        pos = 6 + _u32(data, 1)
    assert data[pos] == 3
    n_reads, n_lanes, width = _u32(data, pos + 5), _u32(data, pos + 9), data[pos + 17] & 0x7f
    t = pos + 22 + n_reads * width
    return np.frombuffer(data[t:t + 2 * n_lanes], dtype=np.uint8).reshape(n_lanes, 2).astype(np.int64)


def greedy_literal(sizes, block_first):
    """The reference's chooser for one model type, literally (model_chooser.rs:168-198, driven per block by
    compressor_block.rs:232-280): no model is active at block start; for every read the first minimum of
    size + (0 if the model is the active one else 2) wins, and a SwitchModel slice precedes the read when it changes."""
    chosen, switched = [], []
    for b in range(len(block_first) - 1):
        cur = -1
        for r in range(int(block_first[b]), int(block_first[b + 1])):
            cost = [int(s) + (0 if k == cur else SWITCH_PENALTY) for k, s in enumerate(sizes[r])]
            best = cost.index(min(cost))
            chosen.append(best)
            switched.append(best != cur)
            cur = best
    return np.asarray(chosen, dtype=np.int64), np.asarray(switched, dtype=bool)


def greedy_choices(sizes, block_first):
    """greedy_literal, fast enough for 500 k reads.  With model k active, k stays iff it beats every earlier candidate
    strictly and no later one beats it (first minimum); otherwise every other candidate pays the same penalty, so the
    choice is the first minimum of the raw sizes (which cannot be k: that one would have stayed).
    sizes: [n_reads, n_cand] forward scores of one type's candidates in provider order -> (chosen, switched)."""
    s = np.asarray(sizes, dtype=np.int64)
    R, K = s.shape
    big = np.iinfo(np.int64).max // 4
    pen = s + SWITCH_PENALTY
    pad = np.full((R, 1), big, dtype=np.int64)
    before = np.minimum.accumulate(np.concatenate([pad, pen[:, :-1]], axis=1), axis=1)                # min over j < k
    after = np.minimum.accumulate(np.concatenate([pen[:, 1:], pad], axis=1)[:, ::-1], axis=1)[:, ::-1]  # min over j > k
    stay = ((s < before) & (s <= after)).tolist()
    first_min = np.argmin(s, axis=1).tolist()
    chosen = np.empty(R, dtype=np.int64)
    switched = np.zeros(R, dtype=bool)
    for b in range(len(block_first) - 1):
        cur = -1
        for r in range(int(block_first[b]), int(block_first[b + 1])):
            best = cur if cur >= 0 and stay[r][cur] else first_min[r]
            chosen[r] = best
            switched[r] = best != cur
            cur = best
    return chosen, switched


def oracle_scores(O, models, reads, rows=None):
    rows = range(reads.n_reads) if rows is None else rows
    out = np.zeros((len(rows), len(models)), dtype=np.int64)
    for i, r in enumerate(rows):
        lo, hi = int(reads.read_off[r]), int(reads.read_off[r + 1])
        for k, m in enumerate(models):
            out[i, k] = O.score_read(m, reads.acids[lo:hi], reads.quals[lo:hi])
    return out


def check_choices(blocks, is_acid, n_acid, sizes, bf):
    """the models in force for every read of the compat blocks == the greedy restatement over `sizes` (acids first)"""
    ca, sa = greedy_choices(sizes[:, :n_acid], bf)
    cq, sq = greedy_choices(sizes[:, n_acid:], bf)
    for b, data in enumerate(blocks):
        r0, r1 = int(bf[b]), int(bf[b + 1])
        ga, gq, gsa, gsq = parse_compat_block(data, is_acid)
        assert len(ga) == r1 - r0, f"block {b}: {len(ga)} Sequence slices for {r1 - r0} reads"
        for name, got, want in (("acid model", ga, ca[r0:r1]), ("q-score model", gq - n_acid, cq[r0:r1]),
                                ("acid switch", gsa, sa[r0:r1]), ("q-score switch", gsq, sq[r0:r1])):
            bad = np.flatnonzero(got != want)
            assert not len(bad), (f"block {b}, read {r0 + bad[0]} (#{bad[0]} of the block): {name} {got[bad[0]]}, "
                                  f"greedy restatement {want[bad[0]]}; {len(bad)} reads differ")
    return int(sa.sum()), int(sq.sum())


def test_greedy_restatement_keeps_the_first_minimum():
    """The fast restatement equals the literal one on small integer scores, where ties and penalty ties are common."""
    rng = np.random.default_rng(5)
    for K in (1, 2, 3, 9, 16):
        sizes = rng.integers(10, 15, size=(3000, K))
        bf = np.asarray([0, 0, 1, 32, 33, 97, 1500, 3000])
        ca, sa = greedy_choices(sizes, bf)
        la, ls = greedy_literal(sizes, bf)
        assert np.array_equal(ca, la) and np.array_equal(sa, ls), K
    # block start: everyone pays the penalty, the first of equals wins; then a tie with the penalty keeps the active model
    chosen, switched = greedy_literal([[5, 5], [5, 3], [5, 2], [9, 9]], [0, 3, 4])
    assert chosen.tolist() == [0, 0, 1, 0] and switched.tolist() == [True, False, True, True]


@pytest.mark.parametrize("block_len", [9000, 40000, BLOCK])
def test_reference_walker_and_greedy_match_oracle(O, model_data, reads_1k, block_len):
    """The two references above, against the oracle's own containers of 1 000 reads with 4 + 4 bundled models."""
    acids = sorted(n for n, md in model_data.items() if md.mtype == O.ACID)[:4]
    quals = sorted(n for n, md in model_data.items() if md.mtype == O.QSCORE)[:4]
    models = [O.Model(model_data[n]) for n in acids + quals]
    idn, st = O.compress(models, reads_1k, max_block_total_len=block_len, include_identifiers=False, return_stats=True)
    version, ids, blocks = split_container(idn)
    assert version == 1 and ids == [m.md.identifier for m in models]
    bf = blocks_of(reads_1k, block_len)
    assert len(blocks) == len(bf) - 1
    n_sa, n_sq = check_choices([d for d, _ in blocks], [True] * 4 + [False] * 4, 4, oracle_scores(O, models, reads_1k), bf)
    assert (n_sa, n_sq) == (st["acid_switches"], st["q_switches"])
    assert n_sa > len(blocks) and n_sq > len(blocks)  # the models do change inside blocks: the check has teeth


# ---- GPU fixtures ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gctx():
    from idencomp_b200 import capi
    ctx = capi.Context(0)
    ctx.set_pipeline_blocks(1 << 16)  # host-pointer calls in one piece: the buckets span the whole batch
    yield ctx
    ctx.close()


def offsets(lens):
    ro = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(np.asarray(lens, dtype=np.uint64), out=ro[1:])
    return ro


def compat_file(models, out):
    return b"IDENCOMP\x01" + bytes([1, 0, len(models)]) + b"".join(m.md.identifier for m in models) + out.tobytes() + b"\x00" * 8


def device_blocks(out, block_off):
    return [out[int(block_off[b]) + 8:int(block_off[b + 1])].tobytes() for b in range(len(block_off) - 1)]


def decode(gctx, out, block_off, crc, handles, mode, reads):
    doff = np.append(block_off[:-1] + 8, block_off[-1]).astype(np.uint64)
    dlen = (block_off[1:] - block_off[:-1] - 8).astype(np.uint32)
    ro, a, q = gctx.decompress_blocks(out, doff, crc, handles, block_len=dlen, mode=mode, reads_cap=reads.n_reads,
                                      symbols_cap=int(reads.read_off[-1]))
    assert np.array_equal(ro, reads.read_off), "decoded read lengths differ"
    assert np.array_equal(a, reads.acids) and np.array_equal(q, reads.quals), "decoded symbols differ"


def native_expect(O, models, reads, bf, lane_syms):
    with ThreadPoolExecutor(THREADS) as ex:  # ctypes releases the GIL
        return list(ex.map(lambda b: O.compress_native_block(models, reads, int(bf[b]), int(bf[b + 1] - bf[b]), lane_syms=lane_syms,
                                                             include_identifiers=False), range(len(bf) - 1)))


def check_native(out, block_off, crc, expect):
    for b, (data, ecrc) in enumerate(expect):
        blk = out[int(block_off[b]):int(block_off[b + 1])].tobytes()
        assert _u32(blk, 0) == len(blk) - 8 == len(data), f"native block {b} length"
        assert blk[8:] == data, f"native block {b} differs"
        assert _u32(blk, 4) == ecrc == int(crc[b]), f"native block {b} crc"


# ---- 1. 9 + 9 candidates on a mixed batch at scale ----------------------------------------------------------------------
@pytest.fixture(scope="module")
def mixed(gctx, O, model_data):
    """Candidates: the acid models of SELECT_PAIRS, then their q-score models.  Reads: a pool per pair drawn on the device
    from the pair's own models, cut into runs of 1-64 reads that are shuffled together, so that the chosen model
    changes inside the switcher's per-lane chunks and across their boundaries; plus one contiguous HiSeq run of
    2.5 x sm_count x 8 x 128 reads (one list-kernel grid is sm_count x 8 x 128 threads)."""
    import torch
    n = len(SELECT_PAIRS)
    names = [PAIRS[p][0] for p in SELECT_PAIRS] + [PAIRS[p][1] for p in SELECT_PAIRS]
    models = [O.Model(model_data[nm]) for nm in names]
    handles = [upload(gctx, O, m) for m in models]
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(20241020)
    runs = []
    for i, p in enumerate(SELECT_PAIRS):
        lo, hi = PAIRS[p][2]
        ro = offsets(rng.integers(lo, hi + 1, size=200 if hi >= 1000 else 5000))
        a, q = synth_on_device(gctx, handles[i], handles[n + i], ro, seed=7000 + i)
        r = 0
        while r < len(ro) - 1:
            k = min(int(rng.integers(1, 65)), len(ro) - 1 - r)
            runs.append((np.diff(ro[r:r + k + 1]), a[int(ro[r]):int(ro[r + k])], q[int(ro[r]):int(ro[r + k])]))
            r += k
    runs = [runs[j] for j in rng.permutation(len(runs))]
    n_long = int(2.5 * sm_count * LIST_CTAS_PER_SM * LIST_THREADS)
    ro = offsets(np.full(n_long, 100))
    a, q = synth_on_device(gctx, handles[0], handles[n], ro, seed=7100)
    runs.insert(len(runs) // 2, (np.diff(ro), a, q))
    reads = O.Reads(offsets(np.concatenate([r[0] for r in runs])), np.concatenate([r[1] for r in runs]),
                    np.concatenate([r[2] for r in runs]), None, None)
    yield dict(models=models, handles=handles, n_acid=n, reads=reads, sm_count=sm_count, bf=blocks_of(reads, BLOCK))
    for h in handles:
        gctx.release_model(h)


def coverage(gctx, handles, pairs):
    """pairs: [n, 2] container model indices of the reads (compat) or lanes (native) -> ({variant: count}, largest bucket)"""
    n_models = len(handles)
    cnt = np.bincount(pairs[:, 0] * n_models + pairs[:, 1], minlength=n_models * n_models)
    per_variant = {}
    for key in np.flatnonzero(cnt):
        v = gctx.kernel_variant(handles[key // n_models], handles[key % n_models])
        per_variant[v] = per_variant.get(v, 0) + int(cnt[key])
    return per_variant, int(cnt.max())


def check_coverage(gctx, mx, pairs, what):
    per_variant, largest = coverage(gctx, mx["handles"], pairs)
    print(f"{what} per kernel variant: {dict(sorted(per_variant.items()))}; largest bucket {largest}")
    n_var = int(gctx.L.idn_gpu_kernel_variant_count())
    missing = [v for v in list(range(n_var)) + [-1] if not per_variant.get(v)]
    assert not missing, f"kernel variants that received no {what}: {missing} ({per_variant})"
    bound = 2 * mx["sm_count"] * LIST_CTAS_PER_SM * LIST_THREADS
    assert largest > bound, f"largest bucket {largest} {what}: the list kernels' stride loop does not run twice ({bound})"


@pytest.mark.gpu
def test_mixed_selection_compat_vs_oracle(gctx, O, mixed):
    """Whole-file compat container of the device == the oracle's, with per-read choices checked first against the
    greedy restatement over the device's own score matrix, and that matrix against the oracle on a sample."""
    mx = mixed
    models, handles, reads, bf, n_acid = mx["models"], mx["handles"], mx["reads"], mx["bf"], mx["n_acid"]
    assert len(bf) - 1 >= 8 and reads.n_reads > 2.5 * mx["sm_count"] * LIST_CTAS_PER_SM * LIST_THREADS
    out, block_off, crc, stats = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, handles)
    sizes = gctx.score((reads.read_off, reads.acids, reads.quals), handles).astype(np.int64)
    sample = np.sort(np.random.default_rng(3).choice(reads.n_reads, size=2000, replace=False))
    want = oracle_scores(O, models, reads, sample)
    bad = np.argwhere(sizes[sample] != want)
    assert not len(bad), f"device score of read {sample[bad[0][0]]} under model {bad[0][1]}: {sizes[sample][tuple(bad[0])]} vs {want[tuple(bad[0])]}"
    is_acid = [True] * n_acid + [False] * (len(models) - n_acid)
    blocks = device_blocks(out, block_off)
    n_sa, n_sq = check_choices(blocks, is_acid, n_acid, sizes, bf)
    assert (n_sa, n_sq) == (stats["acid_switches"], stats["q_switches"])
    ref = O.compress(models, reads, quality=7, include_identifiers=False, threads=THREADS)
    assert compat_file(models, out) == ref, "device container differs from the oracle's"
    pairs = np.concatenate([np.stack(parse_compat_block(d, is_acid)[:2], axis=1) for d in blocks])
    check_coverage(gctx, mx, pairs, "reads")
    decode(gctx, out, block_off, crc, handles, COMPAT, reads)


@pytest.mark.gpu
def test_mixed_selection_native_vs_oracle(gctx, O, mixed):
    """The same batch in the native format with a lane quantum of 64 symbols (about one lane per read): every block ==
    the oracle's, and back."""
    mx = mixed
    models, handles, reads, bf = mx["models"], mx["handles"], mx["reads"], mx["bf"]
    gctx.set_lane_symbols(64)
    try:
        out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, handles, mode=NATIVE)
        check_native(out, block_off, crc, native_expect(O, models, reads, bf, 64))
        lanes = np.concatenate([native_lane_models(d) for d in device_blocks(out, block_off)])
        assert len(lanes) > 0.9 * reads.n_reads
        check_coverage(gctx, mx, lanes, "lanes")
        decode(gctx, out, block_off, crc, handles, NATIVE, reads)
    finally:
        gctx.set_lane_symbols(2048)


# ---- 2. ties and the switch penalty ----------------------------------------------------------------------------------
def twin_of(O, m):
    """A model with another identifier whose quantised tables are those of `m`: one probability moved by one ulp."""
    md = m.md
    table = m.cum_table()
    for c in range(md.n_ctx):
        for s in np.flatnonzero(md.probs[c] > 0):
            probs = md.probs.copy()
            probs[c, s] = np.nextafter(probs[c, s], np.float32(1))
            twin = O.Model(O.ModelData(md.mtype, md.spec_name, probs, md.spec_keys, md.spec_ctx,
                                       O.make_identifier(md.mtype, md.spec_name, probs, md.spec_keys, md.spec_ctx)))
            if np.array_equal(twin.cum_table(), table):
                return twin
    raise AssertionError("no one-ulp twin keeps the quantised table")


@pytest.fixture(scope="module")
def ties(gctx, O, model_data):
    """Models M (HiSeq 2000 pair), their twins T and a third model X per type; reads drawn from M, mostly 100 bp with
    some reads of 600-1500 symbols (cut into several lanes at a lane quantum >= 256)."""
    base = PAIRS["hiseq2000"]
    other = PAIRS["novaseq_human"]
    m = {"Ma": O.Model(model_data[base[0]]), "Mq": O.Model(model_data[base[1]]),
         "Xa": O.Model(model_data[other[0]]), "Xq": O.Model(model_data[other[1]])}
    m["Ta"], m["Tq"] = twin_of(O, m["Ma"]), twin_of(O, m["Mq"])
    h = {k: upload(gctx, O, v) for k, v in m.items()}
    rng = np.random.default_rng(17)
    shapes = [0, 1, 31, 32, 33, 64, 65, 40_000]
    bf = offsets(shapes).astype(np.uint32)
    n = int(bf[-1])
    lens = np.where(rng.random(n) < 0.02, rng.integers(600, 1500, size=n), 100)
    reads = O.synth_reads(m["Ma"], m["Mq"], offsets(lens), 0, 99, 500, threads=THREADS)
    yield m, h, reads, bf
    for v in h.values():
        gctx.release_model(v)


TIE_SETS = {
    "M,T": (["Ma", "Ta"], ["Mq", "Tq"]),
    "T,M": (["Ta", "Ma"], ["Tq", "Mq"]),
    "M,T,X": (["Ma", "Ta", "Xa"], ["Mq", "Tq", "Xq"]),
    "X,T,M": (["Xa", "Ta", "Ma"], ["Xq", "Tq", "Mq"]),
}


@pytest.mark.gpu
def test_twin_models_score_alike(gctx, O, ties):
    m, h, reads, _ = ties
    for a, b in (("Ma", "Ta"), ("Mq", "Tq")):
        assert m[a].md.identifier != m[b].md.identifier
        sa, sb = oracle_scores(O, [m[a], m[b]], reads).T
        assert np.array_equal(sa, sb), f"{b} scores unlike {a}"
    dev = gctx.score((reads.read_off, reads.acids, reads.quals), [h["Ma"], h["Ta"], h["Mq"], h["Tq"]])
    assert np.array_equal(dev[:, 0], dev[:, 1]) and np.array_equal(dev[:, 2], dev[:, 3])


@pytest.mark.gpu
@pytest.mark.parametrize("order", list(TIE_SETS))
def test_ties_keep_the_first_minimum_compat(gctx, O, ties, order):
    """Twins tie on every read; at block start both pay the switch penalty and the first in provider order wins, after
    that the active one wins (no penalty).  Blocks of 0, 1, 31, 32, 33, 64, 65 and 40 000 reads."""
    m, h, reads, bf = ties
    names = TIE_SETS[order][0] + TIE_SETS[order][1]
    models, handles = [m[k] for k in names], [h[k] for k in names]
    n_acid = len(TIE_SETS[order][0])
    out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, handles)
    with ThreadPoolExecutor(THREADS) as ex:
        expect = list(ex.map(lambda b: O.compress_block(models, reads, int(bf[b]), int(bf[b + 1] - bf[b]), include_identifiers=False),
                             range(len(bf) - 1)))
    blocks = device_blocks(out, block_off)
    check_choices(blocks, [True] * n_acid + [False] * n_acid, n_acid, oracle_scores(O, models, reads), bf)
    for b, (data, ecrc, _) in enumerate(expect):
        assert blocks[b] == data and int(crc[b]) == ecrc, f"block {b} ({int(bf[b + 1] - bf[b])} reads) differs"
    decode(gctx, out, block_off, crc, handles, COMPAT, reads)


@pytest.mark.gpu
@pytest.mark.parametrize("lane_syms", [64, 300])
@pytest.mark.parametrize("order", list(TIE_SETS))
def test_ties_keep_the_first_minimum_native(gctx, O, ties, order, lane_syms):
    """Per-lane choice: equal summed scores, first candidate wins (lane_choose_kernel); 300 cuts the long reads."""
    m, h, reads, bf = ties
    names = TIE_SETS[order][0] + TIE_SETS[order][1]
    models, handles = [m[k] for k in names], [h[k] for k in names]
    gctx.set_lane_symbols(lane_syms)
    try:
        out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, handles, mode=NATIVE)
    finally:
        gctx.set_lane_symbols(2048)
    expect = native_expect(O, models, reads, bf, lane_syms)
    if lane_syms >= 256:
        assert any(d and d[17] >> 7 for d, _ in expect), "no read was cut"
    check_native(out, block_off, crc, expect)
    decode(gctx, out, block_off, crc, handles, NATIVE, reads)


# ---- 3. candidate limits and the generic fallback --------------------------------------------------------------------
@pytest.fixture(scope="module")
def many(gctx, O):
    """17 + 17 synthetic models of mixed spec types on ragged reads, acids first."""
    reads = toy_reads(O, 4242, n=600)
    specs = SPEC_NAMES[1:]
    acids = [synthetic_model(O, O.ACID, specs[(3 * i) % len(specs)], reads, 500 + i) for i in range(17)]
    quals = [synthetic_model(O, O.QSCORE, specs[(3 * i + 1) % len(specs)], reads, 600 + i) for i in range(17)]
    ha, hq = [upload(gctx, O, x) for x in acids], [upload(gctx, O, x) for x in quals]
    yield reads, acids, quals, ha, hq
    for x in ha + hq:
        gctx.release_model(x)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [COMPAT, NATIVE], ids=["compat", "native"])
def test_16_plus_16_candidates(gctx, O, many, mode):
    """The most candidates a type may have: the switcher's state arrays are full and the decoder buckets
    16 x 16 pairs of a 32-model list (n_models^2 == 1024).  A 17th model of either type is refused."""
    from idencomp_b200.capi import IdnGpuError
    reads, acids, quals, ha, hq = many
    models, handles = acids[:16] + quals[:16], ha[:16] + hq[:16]
    bf = blocks_of(reads, 6000)
    if mode == COMPAT:
        out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, handles)
        check_choices(device_blocks(out, block_off), [True] * 16 + [False] * 16, 16, oracle_scores(O, models, reads), bf)
        assert compat_file(models, out) == O.compress(models, reads, max_block_total_len=6000, include_identifiers=False)
    else:
        gctx.set_lane_symbols(64)
        try:
            out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, handles, mode=NATIVE)
        finally:
            gctx.set_lane_symbols(2048)
        check_native(out, block_off, crc, native_expect(O, models, reads, bf, 64))
    decode(gctx, out, block_off, crc, handles, mode, reads)
    for too_many in (ha[:17] + hq[:16], ha[:16] + hq[:17]):
        with pytest.raises(IdnGpuError) as e:
            gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, too_many, mode=mode)
        assert e.value.kind == "Unsupported"


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [COMPAT, NATIVE], ids=["compat", "native"])
def test_17_plus_17_container_decodes(gctx, O, many, mode):
    """The oracle writes a container listing 17 + 17 models (the device encoder cannot); decoding it needs more than
    kMaxPairs model pairs, so the device takes the run-time-generic decoder without any environment setting."""
    reads, acids, quals, ha, hq = many
    models, handles = acids + quals, ha + hq
    if mode == COMPAT:
        version, ids, blocks = split_container(O.compress(models, reads, max_block_total_len=6000, include_identifiers=False))
        assert version == 1 and len(ids) == 34
    else:
        bf = blocks_of(reads, 6000)
        blocks = native_expect(O, models, reads, bf, 64)
        assert len({tuple(r) for d, _ in blocks for r in native_lane_models(d)}) > 4  # several pairs in use
    sizes = [len(d) + 8 for d, _ in blocks]
    block_off = offsets(sizes)
    out = np.frombuffer(b"".join(len(d).to_bytes(4, "big") + c.to_bytes(4, "big") + d for d, c in blocks), dtype=np.uint8)
    decode(gctx, out, block_off, np.asarray([c for _, c in blocks], dtype=np.uint32), handles, mode, reads)


@pytest.mark.gpu
def test_selection_without_buckets():
    """IDN_NO_BUCKETS=1 (read once per process) sends every selection call through the run-time-generic kernels; the
    tests above run again in a child process with it set and must give the same bytes."""
    sel = "not without_buckets and not host_mirror"
    env = dict(os.environ, IDN_NO_BUCKETS="1")
    r = subprocess.run([sys.executable, "-m", "pytest", __file__, "-x", "-q", "-m", "gpu", "-k", sel, "-p", "no:cacheprovider"],
                       env=env, capture_output=True, text=True, cwd=str(ROOT))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and " failed" not in r.stdout


# ---- 4. the reference's default path through the host mirror ---------------------------------------------------------
@pytest.fixture(scope="module")
def select4_reads(O, model_data):
    """hiseq100_select4-shaped input: 100 bp reads drawn from ERR174310 + SRR2962693, about ten 4 MiB blocks"""
    am, qm = O.Model(model_data[PAIRS["hiseq2000"][0]]), O.Model(model_data[PAIRS["hiseq2000"][1]])
    return O.synth_reads(am, qm, offsets(np.full(400_000, 100)), 0, 20240601, 500, threads=THREADS)


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["one_device", "two_contexts", "native"])
def test_host_mirror_select4_vs_oracle(O, model_data, select4_reads, how):
    """IdnCompressor(all 22 bundled models, quality 7) keeps 4 + 4 by clustering (not pinned here: the reference's RNG
    has no golden); given that set, the file equals the oracle's byte for byte and decodes back."""
    from idencomp_b200 import capi, host
    reads = select4_reads
    names = sorted(model_data)
    hmodels = [host.Model.load(MODELS / f"{n}.msgpack") for n in names]
    by_id = {model_data[n].identifier: n for n in names}
    kw = {"devices": [0, 0]} if how == "two_contexts" else {"mode": capi.MODE_NATIVE} if how == "native" else {}
    c = host.IdnCompressor(hmodels, quality=7, include_identifiers=False, **kw)
    c.add_batch(reads.read_off, reads.acids, reads.quals)
    idn = c.finish()
    retained = [O.Model(model_data[by_id[i]]) for i in c.retained_models()]
    assert [m.mtype for m in retained] == [O.ACID] * 4 + [O.QSCORE] * 4
    st = c.stats()
    c.close()
    version, ids, blocks = split_container(idn)
    assert ids == [m.md.identifier for m in retained]
    bf = blocks_of(reads, BLOCK)
    assert len(blocks) == len(bf) - 1 >= 9
    if how == "native":  # models are chosen per lane: no SwitchModel slices to count
        assert version == 2
        for b, ((data, crc), (want, wcrc)) in enumerate(zip(blocks, native_expect(O, retained, reads, bf, 2048))):
            assert data == want and crc == wcrc, f"native block {b} differs"
    else:
        assert st["acid_model_switches"] > len(blocks) and st["q_score_model_switches"] > len(blocks)
        assert idn == O.compress(retained, reads, quality=7, include_identifiers=False, threads=THREADS)
    d = host.decompress(hmodels, idn)
    assert np.array_equal(d["read_off"], reads.read_off)
    assert np.array_equal(d["acids"], reads.acids) and np.array_equal(d["quals"], reads.quals)

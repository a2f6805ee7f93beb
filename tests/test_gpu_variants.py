"""Every codec-kernel instantiation the benchmarks launch, and every legal context-spec type, against the CPU oracle.

The codec kernels exist in compile-time-specialised variants per (acid spec type, q-score spec type) pair
(`StaticSpecs` SP0.. in csrc/idn_gpu.cu) next to the run-time-generic ones.  Round 1's tests compared only some of them
with the oracle; this file closes that hole:

* every same-sequencer model pair of the reference's `models/` directory, compat AND native container mode, on reads
  drawn from the pair's own models (so that the real context rows are hit, not the uniform dummy row): the container
  and the CRCs byte for byte against the oracle, the decode of those bytes, and the forward scores; the test asserts
  WHICH kernel variant the pair launches (`idn_gpu_kernel_variant`), and a last test asserts that every variant the
  library holds was covered;
* a small synthetic model for each of the 50 legal spec types (`context_spec.rs:532-599`: dummy + 23 generic + 26 light;
  SURVEY.md counts 49 without `dummy`), as acid and as q-score model,
  through the run-time-generic kernels (uniform and per-read-model variants);
* a model with exactly 65 536 contexts, the reference's limit (`sequence_compressor.rs:209-219`).
"""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from gpu_util import PAIRS, SPEC_NAMES, blocks_of, parse_spec, synth_on_device, synthetic_model, toy_reads, upload

pytestmark = pytest.mark.gpu

COMPAT, NATIVE = 1, 2
BLOCK = 4 * 1024 * 1024

_covered = set()


@pytest.fixture(scope="module")
def gctx():
    from idencomp_b200 import capi
    ctx = capi.Context(0)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def models(gctx, O, model_data):
    """name -> (oracle Model, device handle), uploaded on first use."""
    cache = {}

    def get(name):
        if name not in cache:
            m = O.Model(model_data[name])
            cache[name] = (m, upload(gctx, O, m))
        return cache[name]
    return get


def lengths(lo, hi, total_symbols, seed):
    rng = np.random.default_rng(seed)
    n = int(total_symbols // ((lo + hi) // 2))
    lens = np.full(n, lo, dtype=np.uint64) if lo == hi else rng.integers(lo, hi + 1, size=n, dtype=np.uint64)
    ro = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(lens, out=ro[1:])
    return ro


@pytest.mark.parametrize("mode", [COMPAT, NATIVE], ids=["compat", "native"])
@pytest.mark.parametrize("pair", list(PAIRS))
def test_model_pair_vs_oracle(gctx, O, models, pair, mode):
    """>= 200 k short reads (or ~1 400 long ones) = five blocks with a ragged last one, drawn from the pair's own models:
    the container of the device == the oracle's, byte for byte (compat: the whole .idn file; native: every block),
    and the device decodes it back."""
    an, qn, (lo, hi), variant = PAIRS[pair]
    (am, ha), (qm, hq) = models(an), models(qn)
    assert gctx.kernel_variant(ha, hq) == variant, "the pair does not launch the kernel variant this test is meant to cover"
    ro = lengths(lo, hi, max(4.8 * BLOCK, 201_000 * (lo + hi) // 2 if hi < 1000 else 0), seed=len(pair))
    acids, quals = synth_on_device(gctx, ha, hq, ro, seed=20240601 + len(pair))
    reads = O.Reads(ro, acids, quals, None, None)
    bf = blocks_of(reads, BLOCK)
    nb = len(bf) - 1
    assert nb >= 5 and reads.n_reads >= (200_000 if hi < 1000 else 1000)
    out, block_off, crc, stats = gctx.compress_blocks(ro, acids, quals, bf, [ha, hq], mode=mode)
    if mode == COMPAT:
        ids = am.md.identifier + qm.md.identifier
        idn = b"IDENCOMP\x01" + bytes([1, 0, 2]) + ids + out.tobytes() + b"\x00" * 8
        ref = O.compress([am, qm], reads, max_block_total_len=BLOCK, include_identifiers=False, threads=8)
        assert idn == ref, "device container differs from the oracle's"
    else:
        with ThreadPoolExecutor(8) as ex:  # ctypes releases the GIL
            expect = list(ex.map(lambda b: O.compress_native_block([am, qm], reads, int(bf[b]), int(bf[b + 1] - bf[b]), lane_syms=2048,
                                                                   include_identifiers=False), range(nb)))
        for b, (data, ecrc) in enumerate(expect):
            blk = out[int(block_off[b]):int(block_off[b + 1])].tobytes()
            assert int.from_bytes(blk[0:4], "big") == len(data) and blk[8:] == data, f"native block {b} differs"
            assert int.from_bytes(blk[4:8], "big") == ecrc == int(crc[b])
    # decode side: the same kernels' decoders on those (oracle-identical) bytes
    doff = np.append(block_off[:-1] + 8, block_off[-1]).astype(np.uint64)
    dlen = (block_off[1:] - block_off[:-1] - 8).astype(np.uint32)
    dro, da, dq = gctx.decompress_blocks(out, doff, crc, [ha, hq], block_len=dlen, mode=mode,
                                         reads_cap=reads.n_reads, symbols_cap=int(ro[-1]))
    assert np.array_equal(dro, ro) and np.array_equal(da, acids) and np.array_equal(dq, quals)
    _covered.add((variant, mode))


@pytest.mark.parametrize("pair", list(PAIRS))
def test_model_pair_scores_and_fast_mode(gctx, O, models, pair):
    """forward scores (model_chooser.rs:215-243) and the --fast container (compressor_block.rs:95-106) of a smaller batch"""
    an, qn, (lo, hi), _ = PAIRS[pair]
    (am, ha), (qm, hq) = models(an), models(qn)
    ro = lengths(lo, hi, 300_000, seed=5)
    acids, quals = synth_on_device(gctx, ha, hq, ro, seed=77)
    reads = O.Reads(ro, acids, quals, None, None)
    n = min(reads.n_reads, 64)
    sizes = gctx.score((ro[:n + 1], acids[:int(ro[n])], quals[:int(ro[n])]), [ha, hq])
    for r in range(n):
        s0, s1 = int(ro[r]), int(ro[r + 1])
        assert int(sizes[r, 0]) == O.score_read(am, acids[s0:s1], quals[s0:s1])
        assert int(sizes[r, 1]) == O.score_read(qm, acids[s0:s1], quals[s0:s1])
    bf = blocks_of(reads, 100_000)
    out, block_off, crc, _ = gctx.compress_blocks(ro, acids, quals, bf, [ha, hq], fast=True)
    ref = O.compress([am, qm], reads, max_block_total_len=100_000, include_identifiers=False, fast=True)
    assert out.tobytes() == ref[9 + 3 + 64:-8]


def test_every_specialised_variant_was_compared_with_the_oracle(gctx):
    """runs after the parametrised tests above (pytest keeps file order)"""
    n = int(gctx.L.idn_gpu_kernel_variant_count())
    missing = [(v, m) for v in list(range(n)) + [-1] for m in (COMPAT, NATIVE) if (v, m) not in _covered]
    assert not missing, f"kernel variants never compared with the oracle: {missing}"


# ---- all legal spec types (context_spec.rs:532-599): 1 dummy + 23 generic + 26 light ---------------------------------
@pytest.mark.parametrize("i", range(len(SPEC_NAMES)), ids=SPEC_NAMES)
def test_every_legal_spec_type(gctx, O, i):
    """An acid model of spec type i with a q-score model of spec type i + 7 (so every type serves in both roles across the
    run): container (compat + native), decode and scores against the oracle, through the run-time-generic kernels --
    uniform pair, and per-read selection among two pairs."""
    name_a, name_q = SPEC_NAMES[i], SPEC_NAMES[(i + 7) % len(SPEC_NAMES)]
    assert parse_spec(name_a) and O.spec_num(name_a) >= 1
    reads = toy_reads(O, 100 + i)
    am, qm = synthetic_model(O, O.ACID, name_a, reads, i), synthetic_model(O, O.QSCORE, name_q, reads, 1000 + i)
    am2, qm2 = synthetic_model(O, O.ACID, name_q, reads, 2000 + i), synthetic_model(O, O.QSCORE, name_a, reads, 3000 + i)
    hs = [upload(gctx, O, m) for m in (am, qm, am2, qm2)]
    try:
        bf = blocks_of(reads, 1500)
        for mdl, hd in (([am, qm], [hs[0], hs[1]]), ([am, am2, qm, qm2], [hs[0], hs[2], hs[1], hs[3]])):
            out, block_off, crc, stats = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, hd)
            ids = b"".join(m.md.identifier for m in mdl)
            idn = b"IDENCOMP\x01" + bytes([1, 0, len(mdl)]) + ids + out.tobytes() + b"\x00" * 8
            assert idn == O.compress(mdl, reads, max_block_total_len=1500, include_identifiers=False), (name_a, name_q, len(mdl))
            doff = np.append(block_off[:-1] + 8, block_off[-1]).astype(np.uint64)
            dlen = (block_off[1:] - block_off[:-1] - 8).astype(np.uint32)
            dro, da, dq = gctx.decompress_blocks(out, doff, crc, hd, block_len=dlen)
            assert np.array_equal(dro, reads.read_off) and np.array_equal(da, reads.acids) and np.array_equal(dq, reads.quals)
            gctx.set_lane_symbols(256)
            out2, boff2, crc2, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, hd, mode=NATIVE)
            gctx.set_lane_symbols(2048)
            for b in range(len(bf) - 1):
                want, wcrc = O.compress_native_block(mdl, reads, int(bf[b]), int(bf[b + 1] - bf[b]), lane_syms=256, include_identifiers=False)
                assert out2[int(boff2[b]) + 8:int(boff2[b + 1])].tobytes() == want and int(crc2[b]) == wcrc
            doff = np.append(boff2[:-1] + 8, boff2[-1]).astype(np.uint64)
            dlen = (boff2[1:] - boff2[:-1] - 8).astype(np.uint32)
            dro, da, dq = gctx.decompress_blocks(out2, doff, crc2, hd, block_len=dlen, mode=NATIVE)
            assert np.array_equal(dro, reads.read_off) and np.array_equal(da, reads.acids) and np.array_equal(dq, reads.quals)
        sizes = gctx.score((reads.read_off, reads.acids, reads.quals), hs)
        for r in range(0, reads.n_reads, 5):
            s0, s1 = int(reads.read_off[r]), int(reads.read_off[r + 1])
            for k, m in enumerate((am, qm, am2, qm2)):
                assert int(sizes[r, k]) == O.score_read(m, reads.acids[s0:s1], reads.quals[s0:s1]), (name_a, name_q, r, k)
    finally:
        for h in hs:
            gctx.release_model(h)


def test_model_with_65536_contexts(gctx, O):
    """check_model accepts up to 65 536 contexts (sequence_compressor.rs:209-219); with the dummy row that is 65 537 table
    rows, one more than a u16 row number holds."""
    rng = np.random.default_rng(9)
    n = 65536
    # generic_ao8_qo0_pb0: spec = the last eight acids in base 5, bit-packed below 2^19; one context per spec value
    probs = rng.dirichlet(np.full(5, 0.8), size=n).astype(np.float32)
    keys = np.arange(n, dtype=np.uint32)  # specs 0 .. 65535 = histories that start with two N (0) digits: reachable
    md = O.ModelData(O.ACID, "generic_ao8_qo0_pb0", probs, keys, keys.copy(), O.make_identifier(O.ACID, "generic_ao8_qo0_pb0", probs, keys, keys))
    am = O.Model(md)
    qm = O.Model(O.simple_q_score_model())
    ha, hq = upload(gctx, O, am), upload(gctx, O, qm)
    try:
        seqs = []
        for _ in range(200):
            ln = int(rng.integers(20, 90))
            seqs.append(("", rng.integers(0, 5, size=ln), rng.integers(0, 94, size=ln)))
        # a read whose history walks into the LAST context (spec 65535 = 4,0,4,4,0,2,0,... in base 5 digits, newest lowest)
        digits, v = [], 65535
        while v:
            digits.append(v % 5)
            v //= 5
        seqs.append(("", list(reversed(digits)) + [1, 2, 3], [30] * (len(digits) + 3)))
        reads = O.Reads.from_lists(seqs)
        bf = blocks_of(reads, 4000)
        out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, [ha, hq])
        idn = b"IDENCOMP\x01" + bytes([1, 0, 2]) + am.md.identifier + qm.md.identifier + out.tobytes() + b"\x00" * 8
        assert idn == O.compress([am, qm], reads, max_block_total_len=4000, include_identifiers=False)
        doff = np.append(block_off[:-1] + 8, block_off[-1]).astype(np.uint64)
        dlen = (block_off[1:] - block_off[:-1] - 8).astype(np.uint32)
        dro, da, dq = gctx.decompress_blocks(out, doff, crc, [ha, hq], block_len=dlen)
        assert np.array_equal(da, reads.acids) and np.array_equal(dq, reads.quals)
    finally:
        gctx.release_model(ha)
        gctx.release_model(hq)
    # one context more is refused by the library as by the reference
    from idencomp_b200.capi import IdnGpuError
    cum = np.zeros((n + 2, 6), dtype=np.uint16)
    cum[:] = np.asarray([0, 3277, 6554, 9830, 13107, 16384], dtype=np.uint16)
    with pytest.raises(IdnGpuError) as e:
        gctx.upload_model(O.ACID, 0, 8, 0, 0, 0, cum, np.zeros(1, dtype=np.uint32), np.zeros(1, dtype=np.uint32))
    assert e.value.kind == "Unsupported"

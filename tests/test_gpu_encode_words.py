"""The encoder's read walk in three parts: a head coded position by position down to the first word boundary of the
symbol arrays, an interior coded one 4-byte symbol word per step (word-wide range check, word-wide backward CRC), and a
tail where the pipeline runs off the read.  Every read length up to 40, a few long reads, every read start modulo 16,
arrays of equal and of different alignment, compat and native (reads cut into lane pieces) against the oracle byte for
byte; the block CRCs against the separate CRC pass; an invalid symbol in each of the three parts; and the backward CRC
itself restated on the CPU."""
import os
import subprocess
import sys
import zlib
from pathlib import Path

import numpy as np
import pytest

from gpu_util import PAIRS, blocks_of, synth_on_device, upload

ROOT = Path(__file__).resolve().parent.parent
COMPAT, NATIVE = 1, 2
BLOCK = 20_000
# SP0 (the HiSeq pair of the headline workload), another specialised pair, and the run-time-generic kernels
WORD_PAIRS = ["hiseq2000", "novaseq_cat", "hiseq2500_salmonella"]


# ---- the backward CRC without the data table (CPU) ---------------------------------------------------------------------
def _crc_tables():
    tab = []
    for i in range(256):
        c = i
        for _ in range(8):
            c = (c >> 1) ^ (0xEDB88320 if c & 1 else 0)
        tab.append(c)
    rtop = [0] * 256
    for i in range(256):
        rtop[tab[i] >> 24] = i
    tinv = [((tab[rtop[t]] << 8) & 0xFFFFFFFF) | rtop[t] for t in range(256)]
    return tab, tinv


def _gf2_mul(a, b):  # reflected GF(2) product mod P (x^0 = 0x80000000)
    p = 0
    for _ in range(32):
        if b & 0x80000000:
            p ^= a
        a = (a >> 1) ^ (0xEDB88320 if a & 1 else 0)
        b = (b << 1) & 0xFFFFFFFF
    return p


def _back_crc(acids, quals, tinv, word):
    """crc(acids | quals) from the bytes walked last to first, as the encoder does: byte step B <- Linv(B) ^ b, or per
    group of four, B <- Linv^4(B) ^ w (w = the four bytes as a little-endian word: the first one walked highest)"""
    def linv(b):
        return ((b << 8) & 0xFFFFFFFF) ^ tinv[b >> 24]
    n = len(acids)
    ba = bq = 0
    i = n
    while i > 0:
        if word and i >= 4:
            for _ in range(4):
                ba, bq = linv(ba), linv(bq)
            ba ^= int.from_bytes(bytes(acids[i - 4:i]), "little")
            bq ^= int.from_bytes(bytes(quals[i - 4:i]), "little")
            i -= 4
        else:
            i -= 1
            ba, bq = linv(ba) ^ int(acids[i]), linv(bq) ^ int(quals[i])
    if n == 0:
        return 0
    x1 = 0x80000000
    step = 0x00800000  # x^8
    for _ in range(n):
        x1 = _gf2_mul(x1, step)
    x2 = _gf2_mul(x1, x1)
    return ~(_gf2_mul(x1, bq) ^ _gf2_mul(x2, ba ^ 0xFFFFFFFF)) & 0xFFFFFFFF


def test_backward_crc_needs_no_data_table():
    tab, tinv = _crc_tables()
    assert tinv[0] == 0
    rng = np.random.default_rng(7)
    lens = list(range(0, 24)) + [int(x) for x in rng.integers(24, 2001, size=24)] + [2000]
    for ln in lens:
        a = rng.integers(0, 5, size=ln, dtype=np.uint8)
        q = rng.integers(0, 94, size=ln, dtype=np.uint8)
        ref = zlib.crc32(a.tobytes() + q.tobytes())
        assert _back_crc(a, q, tinv, word=False) == ref, ln
        assert _back_crc(a, q, tinv, word=True) == ref, ln


# ---- device -------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gctx():
    from idencomp_b200 import capi
    ctx = capi.Context(0)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def pairs(gctx, O, model_data):
    out = {}
    for p in WORD_PAIRS:
        an, qn, _, variant = PAIRS[p]
        am, qm = O.Model(model_data[an]), O.Model(model_data[qn])
        ha, hq = upload(gctx, O, am), upload(gctx, O, qm)
        assert gctx.kernel_variant(ha, hq) == variant
        out[p] = (am, qm, ha, hq)
    return out


def _read_off():
    """every length 0..40 three times, interleaved so that reads start at every offset mod 16, and long reads (up to the
    compat format's 10 000)"""
    rng = np.random.default_rng(11)
    lens = [ln for _ in range(3) for ln in rng.permutation(41)] + [10_000, 17, 9_999, 3, 9_998]
    ro = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=ro[1:])
    return ro


def _reads(gctx, O, ha, hq, seed):
    ro = _read_off()
    a, q = synth_on_device(gctx, ha, hq, ro, seed=seed)
    return O.Reads(ro, a, q, None, None)


def _check_compat(gctx, O, am, qm, ha, hq, reads):
    bf = blocks_of(reads, BLOCK)
    out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, [ha, hq])
    ids = am.md.identifier + qm.md.identifier
    idn = b"IDENCOMP\x01" + bytes([1, 0, 2]) + ids + out.tobytes() + b"\x00" * 8
    ref = O.compress([am, qm], reads, max_block_total_len=BLOCK, include_identifiers=False)
    assert idn == ref, "device container differs from the oracle's"
    return bf, crc


@pytest.mark.gpu
@pytest.mark.parametrize("pair", WORD_PAIRS)
def test_compat_every_length_and_offset(gctx, O, pairs, pair, tmp_path):
    am, qm, ha, hq = pairs[pair]
    reads = _reads(gctx, O, ha, hq, seed=300 + len(pair))
    assert {int(r) % 16 for r in reads.read_off[:-1]} == set(range(16))
    bf, crc = _check_compat(gctx, O, am, qm, ha, hq, reads)
    # the block CRCs the encoder computes on the way == those of the separate crc_read_kernel pass (a fresh process: the
    # choice is made when the context is created)
    np.savez(tmp_path / "batch.npz", ro=reads.read_off, a=reads.acids, q=reads.quals, bf=bf)
    names = f"{PAIRS[pair][0]!r}, {PAIRS[pair][1]!r}"
    child = f"""
import sys
import numpy as np
sys.path[:0] = [{str(ROOT)!r}, {str(ROOT / 'tests')!r}]
from idencomp_b200 import capi
from oracle import oracle as O
from gpu_util import upload
d = np.load({str(tmp_path / 'batch.npz')!r})
ctx = capi.Context(0)
h = [upload(ctx, O, O.Model(O.ModelData.load_msgpack({str(ROOT / 'models')!r} + '/' + n + '.msgpack'))) for n in ({names})]
_, _, crc, _ = ctx.compress_blocks(d['ro'], d['a'], d['q'], d['bf'], h)
print(' '.join(str(int(c)) for c in crc))
"""
    env = dict(os.environ, IDN_NO_ENC_CRC="1")
    r = subprocess.run([sys.executable, "-c", child], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert [int(x) for x in r.stdout.split()] == [int(c) for c in crc]


@pytest.mark.gpu
@pytest.mark.parametrize("lane_syms", [64, 300])
@pytest.mark.parametrize("pair", WORD_PAIRS)
def test_native_pieces_every_length_and_offset(gctx, O, pairs, pair, lane_syms):
    am, qm, ha, hq = pairs[pair]
    reads = _reads(gctx, O, ha, hq, seed=400 + len(pair))
    bf = blocks_of(reads, BLOCK)
    gctx.set_lane_symbols(lane_syms)
    try:
        out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, [ha, hq], mode=NATIVE)
    finally:
        gctx.set_lane_symbols(2048)
    for b in range(len(bf) - 1):
        data, ecrc = O.compress_native_block([am, qm], reads, int(bf[b]), int(bf[b + 1] - bf[b]), lane_syms=lane_syms,
                                             include_identifiers=False)
        blk = out[int(block_off[b]):int(block_off[b + 1])].tobytes()
        assert int.from_bytes(blk[0:4], "big") == len(data) and blk[8:] == data, f"native block {b} differs"
        assert int.from_bytes(blk[4:8], "big") == ecrc == int(crc[b])


@pytest.mark.gpu
@pytest.mark.parametrize("shift_a,shift_q", [(0, 4), (3, 11), (5, 5), (15, 15), (9, 0)])
def test_array_alignment(gctx, O, pairs, shift_a, shift_q):
    """Arrays that share their alignment mod 16 (the word path, also when they start off a 16-byte boundary) and arrays
    that do not (the byte reader), through the device entry point that takes any address."""
    import ctypes as C

    import torch
    from idencomp_b200 import capi
    am, qm, ha, hq = pairs["hiseq2000"]
    reads = _reads(gctx, O, ha, hq, seed=500)
    S = int(reads.read_off[-1])
    a_d = torch.zeros(S + 32, dtype=torch.uint8, device="cuda")
    q_d = torch.zeros(S + 32, dtype=torch.uint8, device="cuda")
    a_d[shift_a:shift_a + S] = torch.from_numpy(reads.acids).cuda()
    q_d[shift_q:shift_q + S] = torch.from_numpy(reads.quals).cuda()
    ro_d = torch.from_numpy(reads.read_off.view(np.int64)).cuda()
    bf = blocks_of(reads, BLOCK)
    bf_d = torch.from_numpy(bf.astype(np.int32)).cuda()
    nb = len(bf) - 1
    cap = int(gctx.L.idn_gpu_compress_bound(reads.n_reads, S, nb, 0))
    out_d = torch.zeros(cap + 16, dtype=torch.uint8, device="cuda")
    boff_d = torch.zeros(nb + 1, dtype=torch.int64, device="cuda")
    crc_d = torch.zeros(nb, dtype=torch.int32, device="cuda")
    st_d = torch.zeros(8, dtype=torch.int64, device="cuda")
    b = capi.Batch()
    b.n_reads, b.n_symbols, b.n_blocks = reads.n_reads, S, nb
    b.acids, b.quals = a_d.data_ptr() + shift_a, q_d.data_ptr() + shift_q
    b.read_off, b.block_first_read = ro_d.data_ptr(), bf_d.data_ptr()
    hd = np.asarray([ha, hq], dtype=np.int32)
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    gctx.check(gctx.L.idn_gpu_compress_blocks_dev(gctx.h, C.byref(b), capi.MODE_COMPAT, hd.ctypes.data, 2, 0, None,
                                                  out_d.data_ptr(), cap, boff_d.data_ptr(), crc_d.data_ptr(),
                                                  st_d.data_ptr(), sp))
    torch.cuda.synchronize()
    got = out_d[:int(st_d[0])].cpu().numpy().tobytes()
    ref = O.compress([am, qm], reads, max_block_total_len=BLOCK, include_identifiers=False)
    assert got == ref[9 + 3 + 64:-8]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [COMPAT, NATIVE], ids=["compat", "native"])
@pytest.mark.parametrize("where", ["head", "interior", "tail"])
@pytest.mark.parametrize("which", ["acid", "quality"])
def test_invalid_symbol_in_each_part(gctx, O, pairs, mode, where, which):
    from idencomp_b200.capi import IdnGpuError
    am, qm, ha, hq = pairs["hiseq2000"]
    reads = _reads(gctx, O, ha, hq, seed=600)
    ro = reads.read_off
    r = int(np.flatnonzero(np.diff(ro) == 10_000)[0])  # a long read: head, interior and tail all exist
    s0, s1 = int(ro[r]), int(ro[r + 1])
    pos = {"head": s1 - 1, "interior": (s0 + s1) // 2, "tail": s0 + 1}[where]
    a, q = reads.acids.copy(), reads.quals.copy()
    if which == "acid":
        a[pos] = 5
    else:
        q[pos] = 94
    bf = blocks_of(reads, BLOCK)
    with pytest.raises(IdnGpuError) as e:
        gctx.compress_blocks(ro, a, q, bf, [ha, hq], mode=mode)
    assert e.value.kind == "InvalidSymbol"

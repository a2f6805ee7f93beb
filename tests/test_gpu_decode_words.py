"""The decoders' output writer, payload reader and error reports at every alignment a caller can hand them.

SymWriter picks one of three store regimes from dq = quals_out - acids_out: 16-byte stores of the pending words when
dq = 0 mod 16, plain word stores when dq = 4, 8 or 12 mod 16, byte stores otherwise.  Library calls always decode into
two separate allocations (dq = 0 mod 16), so here both arrays are carved out of one sentinel-filled buffer at every
phase and distance, for the compat and native decoders, uniform and per-read / per-lane model selection, with the block
CRCs checked on every call.  Then the container itself at every phase mod 16 under both slice walks, output capacities
at and one below the totals, stale CRC scratch between calls, the pipelined host call's fallback when a sub-chunk
outgrows its share of the staging, and the rule that a failing call reports the first failing block in file order."""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from gpu_util import PAIRS, blocks_of, parse_compat_block, synth_on_device, upload

ROOT = Path(__file__).resolve().parent.parent
COMPAT, NATIVE = 1, 2
BLOCK = 20_000
SAME = object()      # the encoder's block CRCs
SENT = 0xA5          # never a symbol: acids are 0..4, quality scores 0..93
GAP = 48             # sentinel bytes before, between and after the output arrays (>= 32)
WORD_PAIRS = ["hiseq2000", "novaseq_cat", "hiseq2500_salmonella"]  # SP0, another specialised pair, run-time-generic


# ---- the store regime of SymWriter (idn_kernels.cuh), restated -----------------------------------------------------
def regime(dq):
    """dq & 15 == 0: 16-byte stores; dq & 3 == 0: word stores; otherwise byte stores (Python's % is the two's
    complement residue for negative dq as well)"""
    return "sym16" if dq % 16 == 0 else ("word" if dq % 4 == 0 else "byte")


def layouts(S):
    """(name, acids offset, quals offset, buffer size) in one 16-byte aligned buffer: acids at every phase sa, quals
    after and before them at every residue of dq mod 16, and back to back (dq = S)"""
    out = []
    big = -(-S // 16) * 16 + 3 * GAP
    for sa in range(16):
        for res in range(16):
            dq = S + GAP + (res - S - GAP) % 16                # quals after acids
            out.append((f"sa{sa}+{res}", GAP + sa, GAP + sa + dq))
            dq = -(S + GAP + (-res - S - GAP) % 16)            # quals before acids, dq = res mod 16
            assert dq % 16 == res
            out.append((f"sa{sa}-{res}", big + sa, big + sa + dq))
        out.append((f"sa{sa}=S", GAP + sa, GAP + sa + S))
    size = max(max(a, q) for _, a, q in out) + S + GAP
    return [(n, a, q, size) for n, a, q in out]


def test_layouts_reach_every_regime():
    ro = _read_off()
    S = int(ro[-1])
    lay = layouts(S)
    seen = {regime(q - a) for _, a, q, _ in lay}
    assert seen == {"sym16", "word", "byte"}
    assert {(q - a) % 16 for _, a, q, _ in lay if q > a} == set(range(16))
    assert {(q - a) % 16 for _, a, q, _ in lay if q < a} == set(range(16))
    for _, a, q, size in lay:
        lo, hi = min(a, q), max(a, q)
        assert lo >= GAP and hi - lo >= S and size - (hi + S) >= GAP and (hi - lo - S >= GAP or hi - lo == S)
    # in the 16-byte regime, reads of 16 or more symbols start on a 16-byte boundary: full 16-byte stores happen
    lens = np.diff(ro)
    for _, a, q, _ in lay:
        if regime(q - a) == "sym16":
            assert any((a + int(ro[r])) % 16 == 0 and lens[r] >= 16 for r in range(len(lens)))


# ---- device fixtures -----------------------------------------------------------------------------------------------
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


def _read_off(long_only=False):
    """every length 0..40 three times, interleaved so that reads start at every offset mod 16, and long reads (up to the
    compat format's 10 000); long_only: long reads alone (the warp-per-read CRC pass)"""
    rng = np.random.default_rng(11)
    if long_only:
        lens = [10_000, 9_999, 17, 9_998, 3, 5_001, 10_000, 0, 8_191]
    else:
        lens = [ln for _ in range(3) for ln in rng.permutation(41)] + [10_000, 17, 9_999, 3, 9_998]
    ro = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=ro[1:])
    return ro


def _offsets(lens):
    ro = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=ro[1:])
    return ro


class Enc:
    """a batch, its container from the device encoder, and the decode table (payloads without the 8-byte headers)"""

    def __init__(self, gctx, O, reads, handles, mode, block=BLOCK, bf=None, lane_syms=2048):
        self.reads, self.handles, self.mode = reads, handles, mode
        self.bf = blocks_of(reads, block) if bf is None else np.asarray(bf, dtype=np.uint32)
        gctx.set_lane_symbols(lane_syms)
        try:
            self.out, self.block_off, self.crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, self.bf,
                                                                         handles, mode=mode)
        finally:
            gctx.set_lane_symbols(2048)
        self.nb = len(self.bf) - 1
        self.nbytes = int(self.block_off[-1])
        self.doff = np.append(self.block_off[:-1] + 8, self.nbytes).astype(np.uint64)
        self.dlen = (self.block_off[1:] - self.block_off[:-1] - 8).astype(np.uint32)
        self.R, self.S = reads.n_reads, int(reads.read_off[-1])

    def payload(self, b):
        return self.out[int(self.doff[b]):int(self.doff[b]) + int(self.dlen[b])]

    def host(self, gctx, region=None, crc=SAME, dlen=None, reads_cap=None, symbols_cap=None):
        """idn_gpu_decompress_blocks -> (read_off, acids, quals)"""
        return gctx.decompress_blocks(self.out if region is None else region, self.doff, self.crc if crc is SAME else crc,
                                      self.handles, reads_cap=self.R if reads_cap is None else reads_cap,
                                      symbols_cap=self.S if symbols_cap is None else symbols_cap, mode=self.mode,
                                      block_len=self.dlen if dlen is None else dlen)


class DevIn:
    """the container on the device at base + k, followed by `tail` bytes of `fill`"""

    def __init__(self, enc, k=0, region=None, crc=SAME, dlen=None, tail=64, fill=0):
        import torch
        region = enc.out if region is None else region
        n = enc.nbytes
        self.buf = torch.full((k + n + tail,), fill, dtype=torch.uint8, device="cuda")
        self.buf[k:k + n] = torch.from_numpy(np.ascontiguousarray(region[:n])).cuda()
        self.ptr = self.buf.data_ptr() + k
        self.doff = torch.from_numpy(enc.doff.view(np.int64).copy()).cuda()
        self.dlen = torch.from_numpy((enc.dlen if dlen is None else dlen).view(np.int32).copy()).cuda()
        crc = enc.crc if crc is SAME else crc
        self.crc = None if crc is None else torch.from_numpy(np.asarray(crc, dtype=np.uint32).view(np.int32).copy()).cuda()


def dev_decode(gctx, enc, din, a_ptr, q_ptr, ro_ptr, reads_cap=None, symbols_cap=None):
    """idn_gpu_decompress_blocks_dev -> status_dev [code, block, reads, symbols]"""
    import torch
    st = torch.full((4,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    hd = np.asarray(enc.handles, dtype=np.int32)
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    gctx.check(gctx.L.idn_gpu_decompress_blocks_dev(
        gctx.h, din.ptr, din.doff.data_ptr(), din.dlen.data_ptr(), None if din.crc is None else din.crc.data_ptr(), enc.nb,
        enc.nbytes, enc.mode, hd.ctypes.data, len(hd), a_ptr, q_ptr, ro_ptr, enc.R if reads_cap is None else reads_cap,
        enc.S if symbols_cap is None else symbols_cap, st.data_ptr(), sp))
    torch.cuda.synchronize()
    return st.cpu().tolist()


def _synth(gctx, O, ha, hq, ro, seed):
    a, q = synth_on_device(gctx, ha, hq, ro, seed=seed)
    return O.Reads(ro, a, q, None, None)


def _mixed_reads(gctx, O, pairs, ro, seed):
    """reads drawn alternately from two model pairs, so that per-read / per-lane selection picks both"""
    p0, p1 = pairs["hiseq2000"], pairs["novaseq_cat"]
    a0, q0 = synth_on_device(gctx, p0[2], p0[3], ro, seed=seed)
    a1, q1 = synth_on_device(gctx, p1[2], p1[3], ro, seed=seed + 1)
    a, q = a0.copy(), q0.copy()
    for r in range(1, len(ro) - 1, 2):
        s0, s1 = int(ro[r]), int(ro[r + 1])
        a[s0:s1], q[s0:s1] = a1[s0:s1], q1[s0:s1]
    return O.Reads(ro, a, q, None, None)


# configuration -> (mode, lane quantum, model pair or "select", read lengths)
CONFIGS = {
    "compat_hiseq2000": (COMPAT, 2048, "hiseq2000", False),
    "compat_novaseq_cat": (COMPAT, 2048, "novaseq_cat", False),
    "compat_hiseq2500_salmonella": (COMPAT, 2048, "hiseq2500_salmonella", False),
    "compat_select": (COMPAT, 2048, "select", False),
    "native_q64": (NATIVE, 64, "hiseq2000", False),
    "native_q300": (NATIVE, 300, "hiseq2000", False),
    "native_q300_long": (NATIVE, 300, "hiseq2000", True),
    "native_q2048": (NATIVE, 2048, "hiseq2000", False),
    "native_select": (NATIVE, 300, "select", False),
}


@pytest.fixture(scope="module")
def encoded(gctx, O, pairs):
    cache = {}

    def get(name):
        if name not in cache:
            mode, q, pair, long_only = CONFIGS[name]
            ro = _read_off(long_only)
            if pair == "select":
                reads = _mixed_reads(gctx, O, pairs, ro, seed=900 + len(name))
                p0, p1 = pairs["hiseq2000"], pairs["novaseq_cat"]
                handles = [p0[2], p1[2], p0[3], p1[3]]
            else:
                am, qm, ha, hq = pairs[pair]
                reads = _synth(gctx, O, ha, hq, ro, seed=700 + len(name))
                handles = [ha, hq]
            enc = Enc(gctx, O, reads, handles, mode, lane_syms=q)
            if name == "compat_hiseq2000":  # the container the decoders read is the oracle's
                am, qm = pairs[pair][:2]
                ref = O.compress([am, qm], reads, max_block_total_len=BLOCK, include_identifiers=False)
                ids = am.md.identifier + qm.md.identifier
                assert b"IDENCOMP\x01" + bytes([1, 0, 2]) + ids + enc.out.tobytes() + b"\x00" * 8 == ref
            if name == "compat_select":  # per-read selection really mixes the pairs
                is_acid = [True, True, False, False]
                seen = set()
                for b in range(enc.nb):
                    acid, qual, _, _ = parse_compat_block(enc.payload(b).tobytes(), is_acid)
                    seen |= set(zip(acid.tolist(), qual.tolist()))
                assert len(seen) >= 2, seen
            cache[name] = enc
        return cache[name]
    return get


# ---- A. output writer at every phase --------------------------------------------------------------------------------
def _check_all_layouts(gctx, enc, only=None):
    import torch
    S, R = enc.S, enc.R
    a_t = torch.from_numpy(enc.reads.acids).cuda()
    q_t = torch.from_numpy(enc.reads.quals).cuda()
    ro_want = torch.from_numpy(enc.reads.read_off.view(np.int64).copy()).cuda()
    din = DevIn(enc)
    lay = layouts(S)
    if only is not None:
        lay = lay[::only]
    buf = torch.empty(lay[0][3], dtype=torch.uint8, device="cuda")
    ro = torch.empty(R + 1 + 8, dtype=torch.int64, device="cuda")
    seen = set()
    for i, (name, a_off, q_off, _) in enumerate(lay):
        buf.fill_(SENT)
        ro.fill_(-7)
        with_ro = not name.endswith("=S") or i % 2 == 0  # read_off_out = NULL on some back-to-back calls
        st = dev_decode(gctx, enc, din, buf.data_ptr() + a_off, buf.data_ptr() + q_off, ro.data_ptr() if with_ro else None)
        assert st == [0, -1, R, S], f"{name}: status {st}"
        want = torch.full_like(buf, SENT)
        want[a_off:a_off + S] = a_t
        want[q_off:q_off + S] = q_t
        if not torch.equal(buf, want):
            bad = torch.nonzero(buf != want).flatten()[:8].tolist()
            pytest.fail(f"{name} ({regime(q_off - a_off)} stores): bytes differ at buffer offsets {bad}")
        if with_ro:
            assert torch.equal(ro[:R + 1], ro_want), name
            assert bool((ro[R + 1:] == -7).all()), name
        else:
            assert bool((ro == -7).all()), name
        seen.add(regime(q_off - a_off))
    assert seen == {"sym16", "word", "byte"}


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
def test_output_every_phase(gctx, encoded, config):
    """Every acids phase mod 16, quals after and before the acids at every residue of dq mod 16, and back to back: the
    symbols, the read offsets, the status words and every sentinel byte around and between the arrays."""
    _check_all_layouts(gctx, encoded(config))


@pytest.mark.gpu
def test_selection_output_without_buckets():
    """IDN_NO_BUCKETS=1 (read once per process) sends the selection decodes through the run-time-generic kernels"""
    env = dict(os.environ, IDN_NO_BUCKETS="1")
    r = subprocess.run([sys.executable, "-m", "pytest", __file__, "-x", "-q", "-m", "gpu", "-k", "test_output_every_phase and select",
                        "-p", "no:cacheprovider"], env=env, capture_output=True, text=True, cwd=str(ROOT), timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "2 passed" in r.stdout


# ---- B. payload reader and slice walks at every buffer alignment ---------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("config", ["compat_hiseq2000", "compat_select", "native_q300", "native_q2048"])
def test_container_every_phase(gctx, encoded, config):
    """The container at device base + k for k = 0..15 with its region ending at its last byte, under both slice walks,
    with the bytes after the region 0x00 or 0xFF: every payload starts at every phase mod 4 and the walks stage
    unaligned buffer ends."""
    import torch
    enc = encoded(config)
    S, R = enc.S, enc.R
    a_t = torch.from_numpy(enc.reads.acids).cuda()
    q_t = torch.from_numpy(enc.reads.quals).cuda()
    ro_want = torch.from_numpy(enc.reads.read_off.view(np.int64).copy()).cuda()
    a = torch.empty(S + 16, dtype=torch.uint8, device="cuda")
    q = torch.empty(S + 16, dtype=torch.uint8, device="cuda")
    ro = torch.empty(R + 1, dtype=torch.int64, device="cuda")
    walks = (1, 2) if enc.mode == COMPAT else (0,)
    try:
        for k in range(16):
            for fill in (0x00, 0xFF):
                din = DevIn(enc, k=k, fill=fill)
                assert din.ptr % 16 == k
                for w in walks:
                    gctx.set_walk(w)
                    a.fill_(SENT)
                    q.fill_(SENT)
                    st = dev_decode(gctx, enc, din, a.data_ptr(), q.data_ptr(), ro.data_ptr())
                    assert st == [0, -1, R, S], (k, fill, w, st)
                    assert torch.equal(a[:S], a_t) and torch.equal(q[:S], q_t) and torch.equal(ro, ro_want), (k, fill, w)
                    assert bool((a[S:] == SENT).all()) and bool((q[S:] == SENT).all())
    finally:
        gctx.set_walk(0)


# ---- C. capacities and stale scratch ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("config", ["compat_hiseq2000", "native_q300", "native_q2048"])
def test_capacities(gctx, encoded, config):
    import torch
    from idencomp_b200.capi import IdnGpuError
    enc = encoded(config)
    S, R = enc.S, enc.R
    din = DevIn(enc)
    a = torch.empty(S + GAP, dtype=torch.uint8, device="cuda")
    q = torch.empty(S + GAP, dtype=torch.uint8, device="cuda")
    ro = torch.empty(R + 1 + 4, dtype=torch.int64, device="cuda")
    for rc, sc in [(R, S), (R - 1, S), (R, S - 1), (R - 1, S - 1)]:
        a.fill_(SENT)
        q.fill_(SENT)
        ro.fill_(-7)
        st = dev_decode(gctx, enc, din, a.data_ptr(), q.data_ptr(), ro.data_ptr(), reads_cap=rc, symbols_cap=sc)
        if (rc, sc) == (R, S):
            assert st == [0, -1, R, S]
            assert bool((a[S:] == SENT).all()) and bool((q[S:] == SENT).all()) and bool((ro[R + 1:] == -7).all())
            assert np.array_equal(a[:S].cpu().numpy(), enc.reads.acids)
            continue
        assert st[:3] == [11, -1, R], (rc, sc, st)  # NoSpace, the read count the call needs
        assert bool((a == SENT).all()) and bool((q == SENT).all()), "a call that fails wrote symbols"
    # host-pointer calls: the same shortfalls at every sub-chunk size
    try:
        for pb in (1, 3, 1000):
            gctx.set_pipeline_blocks(pb)
            ro_h, a_h, q_h = enc.host(gctx)
            assert np.array_equal(ro_h, enc.reads.read_off) and np.array_equal(a_h, enc.reads.acids)
            assert np.array_equal(q_h, enc.reads.quals)
            for rc, sc in [(R - 1, S), (R, S - 1)]:
                with pytest.raises(IdnGpuError) as e:
                    enc.host(gctx, reads_cap=rc, symbols_cap=sc)
                assert e.value.kind == "NoSpace", (pb, rc, sc)
    finally:
        gctx.set_pipeline_blocks(32)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [COMPAT, NATIVE], ids=["compat", "native"])
def test_empty_reads_after_a_large_call(gctx, O, pairs, mode):
    """Blocks that start and end with empty reads, and a block of empty reads only, decoded right after a larger call on
    the same context: no per-read CRC partial of the earlier call may leak into the block CRCs."""
    from idencomp_b200 import capi
    am, qm, ha, hq = pairs["hiseq2000"]
    ctx = capi.Context(0)
    try:
        h = [upload(ctx, O, am), upload(ctx, O, qm)]
        big = Enc(ctx, O, _synth(gctx, O, ha, hq, _offsets(np.full(30_000, 100)), seed=31), h, mode)
        ro, a, q = big.host(ctx)
        assert np.array_equal(a, big.reads.acids)
        lens = [0, 0, 57, 16, 0, 0, 33, 0] + [0] * 9 + [0, 1, 200, 0]
        bf = [0, 8, 17, len(lens)]
        small = Enc(ctx, O, _synth(gctx, O, ha, hq, _offsets(lens), seed=32), h, mode, bf=bf)
        ro, a, q = small.host(ctx)
        assert np.array_equal(ro, small.reads.read_off) and np.array_equal(a, small.reads.acids)
        assert np.array_equal(q, small.reads.quals)
        import torch
        din = DevIn(small)
        at = torch.zeros(small.S + 16, dtype=torch.uint8, device="cuda")
        qt = torch.zeros(small.S + 16, dtype=torch.uint8, device="cuda")
        rt = torch.zeros(small.R + 1, dtype=torch.int64, device="cuda")
        assert dev_decode(ctx, small, din, at.data_ptr(), qt.data_ptr(), rt.data_ptr()) == [0, -1, small.R, small.S]
    finally:
        ctx.close()


# ---- D. the pipelined decode's fallback ------------------------------------------------------------------------------
def sub_chunk_overflows(doff, dlen, bf_syms, bf_reads, sub, reads_cap, syms_cap):
    """decompress_blocks_pipelined (idn_pipeline.inc): a sub-chunk's staging holds min(cap, share * 1.25 * cap + margin)
    symbols (margin 8 MiB) and reads (margin 64 Ki), share = its container bytes over the region's; True if some
    sub-chunk needs more (the call then decodes unpipelined)"""
    nb = len(dlen)
    total = float(doff[-1])
    for b0 in range(0, nb, sub):
        b1 = min(nb, b0 + sub)
        share = (float(doff[b1 - 1]) + float(dlen[b1 - 1]) - float(doff[b0])) / total
        cap_s = min(syms_cap, int(share * 1.25 * syms_cap) + (8 << 20))
        cap_r = min(reads_cap, int(share * 1.25 * reads_cap) + (1 << 16))
        if bf_syms[b1] - bf_syms[b0] > cap_s or bf_reads[b1] - bf_reads[b0] > cap_r:
            return True
    return False


def test_sub_chunk_rule_restated():
    doff = np.asarray([0, 100, 200, 300, 400], dtype=np.uint64)
    dlen = np.full(4, 100, dtype=np.uint32)
    even = np.asarray([0, 1, 2, 3, 4]) * (4 << 20)
    assert not sub_chunk_overflows(doff, dlen, even, np.arange(5), 1, 4, 16 << 20)
    skew = np.asarray([0, 1, 2, 3, 20]) * (1 << 20)  # the last block: 17 Mi symbols in a quarter of the bytes
    assert sub_chunk_overflows(doff, dlen, skew, np.arange(5), 1, 4, 20 << 20)
    assert not sub_chunk_overflows(doff, dlen, skew, np.arange(5), 4, 4, 20 << 20)


def _peaked_model(O, mtype, sym):
    """a model without context (spec type dummy) that gives `sym` all but the least frequency the quantiser allows"""
    key = O.Generator("dummy", 1).current_context()
    n = 5 if mtype == O.ACID else 94
    p = np.full(n, 1e-7, dtype=np.float64)
    p[sym] = 1.0 - 1e-7 * (n - 1)
    return O.Model(O.ModelData.from_contexts(mtype, "dummy", [([key], p.tolist())]))


@pytest.mark.gpu
def test_pipelined_fallback(gctx, O):
    """Runs of blocks of random symbols (several bytes per symbol under a peaked model) and runs of blocks of the model's
    favourite symbols (a few bytes per thousand symbols): with 4 blocks per sub-chunk a constant sub-chunk needs far more
    symbols than its share of the container bytes gives it, and the call falls back to the unpipelined decode."""
    ha, hq = upload(gctx, O, _peaked_model(O, O.ACID, 2)), upload(gctx, O, _peaked_model(O, O.QSCORE, 37))
    rng = np.random.default_rng(5)
    L = 1000
    runs = [("rand", 1_000_000), ("const", 3_000_000), ("rand", 1_000_000), ("const", 3_000_000), ("rand", 1_000_000)]
    a_parts, q_parts, bf, n = [], [], [0], 0
    for kind, per_block in runs:
        for _ in range(4):
            k = per_block // L
            if kind == "rand":
                a_parts.append(rng.integers(0, 5, size=k * L, dtype=np.uint8))
                q_parts.append(rng.integers(0, 94, size=k * L, dtype=np.uint8))
            else:
                a_parts.append(np.full(k * L, 2, dtype=np.uint8))
                q_parts.append(np.full(k * L, 37, dtype=np.uint8))
            n += k
            bf.append(n)
    acids, quals = np.concatenate(a_parts), np.concatenate(q_parts)
    reads = O.Reads(_offsets(np.full(n, L)), acids, quals, None, None)
    enc = Enc(gctx, O, reads, [ha, hq], COMPAT, bf=bf)
    bf_syms = np.asarray(bf, dtype=np.int64) * L
    assert not sub_chunk_overflows(enc.doff, enc.dlen, bf_syms, np.asarray(bf), 1 << 30, enc.R, enc.S)
    assert sub_chunk_overflows(enc.doff, enc.dlen, bf_syms, np.asarray(bf), 4, enc.R, enc.S), \
        f"the constant runs ({int(enc.dlen[4])} bytes per block) do not overflow their share"
    try:
        gctx.set_pipeline_blocks(4)
        ro, a, q = enc.host(gctx)
    finally:
        gctx.set_pipeline_blocks(32)
        gctx.release_model(ha)
        gctx.release_model(hq)
    assert np.array_equal(ro, reads.read_off) and np.array_equal(a, acids) and np.array_equal(q, quals)


# ---- E. the first failing block in file order ------------------------------------------------------------------------
def reports(gctx, enc, region=None, crc=SAME, dlen=None):
    """(error kind, block) of the _dev call under both walks and of the host-pointer call at sub-chunks of 1, 3 and 1000
    blocks under both walks"""
    from idencomp_b200.capi import ERRORS, IdnGpuError
    import torch
    out = {}
    din = DevIn(enc, region=region, crc=crc, dlen=dlen)
    a = torch.empty(enc.S + 16, dtype=torch.uint8, device="cuda")
    q = torch.empty(enc.S + 16, dtype=torch.uint8, device="cuda")
    ro = torch.empty(enc.R + 1, dtype=torch.int64, device="cuda")
    try:
        for w in (1, 2):
            gctx.set_walk(w)
            st = dev_decode(gctx, enc, din, a.data_ptr(), q.data_ptr(), ro.data_ptr())
            out[f"dev walk {w}"] = (ERRORS[st[0]], st[1])
            for pb in (1, 3, 1000):
                gctx.set_pipeline_blocks(pb)
                try:
                    enc.host(gctx, region=region, crc=crc, dlen=dlen)
                    out[f"host walk {w} sub {pb}"] = ("Ok", -1)
                except IdnGpuError as e:
                    out[f"host walk {w} sub {pb}"] = (e.kind, e.bad_block)
    finally:
        gctx.set_walk(0)
        gctx.set_pipeline_blocks(32)
    return out


def assert_reports(got, want):
    wrong = {k: v for k, v in got.items() if v != want}
    assert not wrong, f"expected {want}, got {wrong}"


@pytest.fixture(scope="module")
def small_blocks(gctx, O, pairs):
    """15 blocks of 200 reads of 100 symbols, compat and native"""
    am, qm, ha, hq = pairs["hiseq2000"]
    reads = _synth(gctx, O, ha, hq, _offsets(np.full(3000, 100)), seed=77)
    return {m: Enc(gctx, O, reads, [ha, hq], m) for m in (COMPAT, NATIVE)}


def _splice(enc, new_payloads):
    """a region with block b's payload replaced by new_payloads[b] (the others as they are) -> (region, dlen)"""
    region = enc.out.copy()
    dlen = enc.dlen.copy()
    for b, data in new_payloads.items():
        assert len(data) <= int(enc.dlen[b]) or b == enc.nb - 1
        lo = int(enc.doff[b])
        region[lo:lo + len(data)] = np.frombuffer(data, dtype=np.uint8)
        dlen[b] = len(data)
    return region, dlen


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [COMPAT, NATIVE], ids=["compat", "native"])
def test_first_block_wins_the_walk_race(gctx, O, pairs, mode):
    """Block 0 holds about 4 Mi symbols and its defect sits at its end, so its walk finishes last; blocks 1.. are small
    and malformed from their first byte.  The report is block 0 and its own error kind, whichever walk finishes first."""
    am, qm, ha, hq = pairs["hiseq2000"]
    n0, n_small = 42_000, 40
    lens = np.concatenate([np.full(n0, 100), np.full(20 * n_small, 100)])
    reads = _synth(gctx, O, ha, hq, _offsets(lens), seed=88)
    bf = np.concatenate([[0], n0 + 20 * np.arange(n_small + 1)]).astype(np.uint32)
    enc = Enc(gctx, O, reads, [ha, hq], mode, bf=bf)
    region = enc.out.copy()
    dlen = enc.dlen.copy()
    lo0 = int(enc.doff[0])
    if mode == COMPAT:
        # block 0 ends with a SwitchModel slice of an index past the model list: the slice replaces the last 2 payload
        # bytes of the block's last read, whose Sequence slice then ends early -- so shorten the block by its last read
        _, _, _, _, p_off, p_len, _ = parse_compat_block(enc.payload(0).tobytes(), [True, False], offsets=True)
        last_hdr = int(p_off[-1]) - 9
        region[lo0 + last_hdr:lo0 + last_hdr + 2] = [1, 9]
        dlen[0] = last_hdr + 2
        want = ("InvalidModelIndex", 0)
    else:
        # block 0: the last lane's q-score model index points past the model list
        body = enc.payload(0).tobytes()
        assert body[0] == 3
        n_reads, n_lanes = int.from_bytes(body[5:9], "big"), int.from_bytes(body[9:13], "big")
        width = body[17] & 0x7F
        fixed = 22
        t_mdl = fixed + n_reads * width
        region[lo0 + t_mdl + 2 * (n_lanes - 1) + 1] = 9
        want = ("InvalidModelIndex", 0)
    for b in range(1, enc.nb):  # an unknown slice kind first
        region[int(enc.doff[b])] = 7
    assert_reports(reports(gctx, enc, region=region, dlen=dlen), want)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [COMPAT, NATIVE], ids=["compat", "native"])
def test_stream_error_names_its_block(gctx, small_blocks, mode):
    """Payload bytes of block 3 garbled with the slice headers intact and no block CRCs: SerializeError in block 3."""
    enc = small_blocks[mode]
    region = enc.out.copy()
    lo = int(enc.doff[3])
    if mode == COMPAT:
        _, _, _, _, p_off, p_len, _ = parse_compat_block(enc.payload(3).tobytes(), [True, False], offsets=True)
        r = int(np.argmax(p_len))
        p = lo + int(p_off[r]) + int(p_len[r]) // 2
    else:
        p = lo + int(enc.dlen[3]) * 3 // 4  # inside the lane payloads, behind the tables
    region[p:p + 4] ^= np.uint8(0x5B)
    assert_reports(reports(gctx, enc, region=region, crc=None), ("SerializeError", 3))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [COMPAT, NATIVE], ids=["compat", "native"])
def test_checksum_before_a_later_malformed_block(gctx, small_blocks, mode):
    """A wrong header CRC in block 2 and a malformed block 5: the checksum mismatch of block 2 is reported."""
    enc = small_blocks[mode]
    region = enc.out.copy()
    region[int(enc.doff[5])] = 7
    crc = enc.crc.copy()
    crc[2] ^= 1
    assert_reports(reports(gctx, enc, region=region, crc=crc), ("BlockChecksumMismatch", 2))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [COMPAT, NATIVE], ids=["compat", "native"])
def test_first_of_several_checksum_mismatches(gctx, small_blocks, mode):
    enc = small_blocks[mode]
    crc = enc.crc.copy()
    for b in (9, 2, 5):
        crc[b] ^= 0x80000000
    assert_reports(reports(gctx, enc, crc=crc), ("BlockChecksumMismatch", 2))

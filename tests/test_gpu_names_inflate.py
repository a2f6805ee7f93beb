"""Identifiers slices inflated on the device (csrc/idn_inflate.cuh, idn_gpu_inflate_names, IdnDecompressor with
identifiers_on_device): every slice zlib's raw inflate accepts must give zlib's bytes, split into names as the host's
inflate_names splits them; every slice zlib rejects must fail with Serialize on its block; the parallel decode must really
join speculative chunks; and the host mirror must read every container exactly as it does with the host's zlib."""
import random
import zlib

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from idencomp_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def bench_titles(n, first=0):
    return [b"r%012d 1:N:0" % i for i in range(first, first + n)]


def illumina_names(n, seed=1):
    rng = random.Random(seed)
    x, y, out = 1000, 1000, []
    for _ in range(n):
        x += rng.randint(1, 40)
        if x > 32000:
            x, y = 1000, y + rng.randint(1, 300)
        out.append(b"A00123:8:H5TJ3DSXX:1:1101:%d:%d 1:N:0:ACGTACGT+TTGCAGGA" % (x, y))
    return out


def slice_rec(data, comp=1):
    return b"\x00" + len(data).to_bytes(4, "big") + bytes([comp]) + data


def zraw(text, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, mem=8, flush_every=0, flush=zlib.Z_SYNC_FLUSH):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, mem, strategy)
    if not flush_every:
        return c.compress(text) + c.flush()
    out = b""
    for i in range(0, len(text), flush_every):
        out += c.compress(text[i:i + flush_every]) + c.flush(flush)
    return out + c.flush()


def zlib_accepts(data):
    """what the host's inflate_raw does: None when it rejects the stream"""
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(data)
    except zlib.error:
        return None
    return out if d.eof else None


def host_split(texts, want):
    """inflate_names of one block: its slices' texts joined with '\\n', at most `want` lines, missing lines empty"""
    if not texts:
        return [b""] * want
    lines = b"\n".join(texts).split(b"\n")[:want]
    return lines + [b""] * (want - len(lines))


def run(ctx, blocks, wants, **kw):
    """blocks: list of payloads (slice records, maybe followed by other bytes) -> names per read and the stats"""
    payload = b"".join(blocks)
    off = np.zeros(len(blocks) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(b) for b in blocks])
    bf = np.zeros(len(blocks) + 1, dtype=np.uint32)
    bf[1:] = np.cumsum(wants)
    names, no, st = ctx.inflate_names(np.frombuffer(payload, dtype=np.uint8), off, bf, **kw)
    nb = names.tobytes()
    return [nb[int(no[r]):int(no[r + 1])] for r in range(len(no) - 1)], st


def check(ctx, block_texts, wants, block_payloads=None):
    """block_texts[b]: list of raw Deflate streams of block b's slices"""
    payloads = block_payloads or [b"".join(slice_rec(s) for s in streams) for streams in block_texts]
    got, st = run(ctx, payloads, wants)
    want = []
    for streams, w in zip(block_texts, wants):
        want += host_split([zlib_accepts(s) for s in streams], w)
    assert got == want
    return st


# ---- 1. streams from zlib -----------------------------------------------------------------------------------------------
TEXT = b"\n".join(bench_titles(30_000))
ILL = b"\n".join(illumina_names(20_000))
RUN258 = b"a" * 70_000 + b"\n" + bytes(range(256)) * 300


@pytest.mark.parametrize("name,stream", [
    ("level0", zraw(TEXT[:200_000], 0)), ("level1", zraw(TEXT, 1)), ("level6", zraw(TEXT, 6)), ("level9", zraw(ILL, 9)),
    ("fixed", zraw(ILL, 6, zlib.Z_FIXED)), ("huffman_only", zraw(TEXT, 6, zlib.Z_HUFFMAN_ONLY)), ("rle", zraw(RUN258, 6, zlib.Z_RLE)),
    ("mem1", zraw(ILL, 6, mem=1)), ("mem9", zraw(ILL, 6, mem=9)), ("sync_flush", zraw(TEXT, 6, flush_every=3000)),
    ("full_flush", zraw(ILL, 6, flush_every=5000, flush=zlib.Z_FULL_FLUSH)), ("empty", zraw(b"")),
    ("window_edges", zraw(b"\n".join(b"x" * n for n in (32767, 32768, 32769, 65535, 65536, 65537)))),
    ("run_d1_l258", zraw(RUN258, 9)), ("all_bytes", zraw(bytes(range(256)) * 500, 6)),
])
def test_zlib_streams(ctx, name, stream):
    text = zlib_accepts(stream)
    assert text is not None
    n = text.count(b"\n") + 1
    for want in (n, n + 3, max(1, n // 2)):
        check(ctx, [[stream]], [want])


def test_large_expansion_and_4mib_block(ctx):
    # ~1000:1 outgrows the first scratch; the call measures and retries inside itself
    run_1m = zraw(b"z" * 1_000_000, 9)
    assert len(run_1m) < 2000
    check(ctx, [[run_1m]], [1])
    big = b"\n".join(illumina_names(80_000, seed=7))
    assert len(big) > 4 << 20
    check(ctx, [[zraw(big, 6)], [run_1m]], [80_000, 2])


def test_device_encoder_slices(ctx):
    for n in (1, 2, 14, 15):
        names = illumina_names(n * 1100, seed=n)  # ~66 bytes per name: n 64 KiB segments
        off = np.zeros(len(names) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(x) for x in names])
        out, so = ctx.deflate_names(off, np.frombuffer(b"".join(names), dtype=np.uint8), np.array([0, len(names)], dtype=np.uint32))
        s = out.tobytes()
        assert zlib_accepts(s[6:]) == b"\n".join(names)
        check(ctx, [[s[6:]]], [len(names)])


# ---- 2. the parallel path runs --------------------------------------------------------------------------------------------
def test_zlib6_blocks_join_chunks(ctx):
    per = 41_943
    streams = [zraw(b"\n".join(bench_titles(per, b * per)), 6) for b in range(4)]
    st = check(ctx, [[s] for s in streams], [per] * 4)
    assert st["n_streams"] == 4
    assert st["n_joined"] > 4, st  # more than one chunk per stream on average joins
    assert st["n_joined"] <= st["n_speculative"]


def test_device_encoder_joins_one_chunk_per_segment(ctx):
    names = bench_titles(41_943 * 2)
    off = np.zeros(len(names) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(x) for x in names])
    out, so = ctx.deflate_names(off, np.frombuffer(b"".join(names), dtype=np.uint8), np.array([0, 41_943, len(names)], dtype=np.uint32))
    s = out.tobytes()
    segs_per_block = -(-(41_943 * 20 - 1) // 65536)
    ctx.set_inflate_range(2048)
    try:
        st = check(ctx, [[s[6:int(so[1])]], [s[int(so[1]) + 6:]]], [41_943, 41_943])
    finally:
        ctx.set_inflate_range(4096)
    assert st["n_joined"] >= 2 * (segs_per_block - 1), st


# ---- 3. false candidates --------------------------------------------------------------------------------------------------
def test_false_candidates(ctx):
    fake = b"\n".join(b"n%05d\x00\x00\xff\xff%s" % (i, b"q" * (i % 90)) for i in range(3000))
    hdr = zraw(ILL[:20000], 6)[:200]  # the bytes of a real dynamic-block header, stored as data
    rnd = np.random.default_rng(5).integers(0, 256, size=300_000, dtype=np.uint8).tobytes()
    ctx.set_inflate_range(1024)
    try:
        st = check(ctx, [[zraw(fake, 0)], [zraw(hdr * 400, 0)], [zraw(rnd, 6)]], [3000, 5, 7])
    finally:
        ctx.set_inflate_range(4096)
    assert st["serial_bytes"] > 0, st


# ---- 4. malformed slices ------------------------------------------------------------------------------------------------
class Bits:
    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, x, k):  # k bits of x, LSB first
        self.v |= (x & ((1 << k) - 1)) << self.n
        self.n += k

    def code(self, c, k):  # a Huffman code, MSB first
        for i in range(k - 1, -1, -1):
            self.put((c >> i) & 1, 1)

    def bytes(self):
        return self.v.to_bytes((self.n + 7) // 8, "little")


def canon(lens):
    codes, code, nxt = {}, 0, [0] * 17
    bl = [0] * 17
    for l in lens:
        bl[l] += 1
    bl[0] = 0
    for b in range(1, 16):
        code = (code + bl[b - 1]) << 1
        nxt[b] = code
    for s, l in enumerate(lens):
        if l:
            codes[s] = (nxt[l], l)
            nxt[l] += 1
    return codes


def fixed_lit(b, s):
    if s < 144:
        b.code(0x30 + s, 8)
    elif s < 256:
        b.code(0x190 + s - 144, 9)
    elif s < 280:
        b.code(s - 256, 7)
    else:
        b.code(0xC0 + s - 280, 8)


def dynamic(lit, dist, syms, cl=None, cl_seq=None, final=1):
    """a dynamic block: lit / dist code lengths, sent with code-length code `cl` (default: 0..15 at 4 bits), then symbols
    (('l', sym) or ('m', lensym, lenextra_bits, distsym, distextra_bits))"""
    b = Bits()
    b.put(final, 1)
    b.put(2, 2)
    b.put(len(lit) - 257, 5)
    b.put(len(dist) - 1, 5)
    cl = cl or ([4] * 16 + [0, 0, 0])
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
    b.put(15, 4)
    for i in range(19):
        b.put(cl[order[i]], 3)
    clc = canon(cl)
    for v in (cl_seq if cl_seq is not None else list(lit) + list(dist)):
        b.code(*clc[v])
    lc, dc = canon(lit), canon(dist)
    for s in syms:
        b.code(*lc[s])
    return b.bytes()


def fixed_block(syms, final=1):
    b = Bits()
    b.put(final, 1)
    b.put(1, 2)
    for s in syms:
        if isinstance(s, tuple):  # (lensym, extra, nextra, distsym, dextra, ndextra)
            fixed_lit(b, s[0])
            b.put(s[1], s[2])
            b.code(s[3], 5)
            b.put(s[4], s[5])
        else:
            fixed_lit(b, s)
    return b.bytes()


def _lens(pairs, n):
    v = [0] * n
    for s, l in pairs.items():
        v[s] = l
    return v


MALFORMED = {
    "btype3": bytes([0b111]),
    "stored_len_nlen": bytes([1, 5, 0, 0, 0]) + b"hello",
    "stored_ok": bytes([1, 5, 0, 0xFA, 0xFF]) + b"hello",
    "oversubscribed": dynamic([8] * 286, [1], []),
    "incomplete": dynamic(_lens({65: 2, 66: 2, 256: 2}, 257), [1, 1], [65, 256]),
    "single_code": dynamic(_lens({256: 1}, 257), [0], [256]),
    "single_dist_code": dynamic(_lens({65: 1, 256: 1}, 257), [1], [65, 65, 256]),
    "no_dist_codes": dynamic(_lens({97: 1, 256: 1}, 257), [0], [97, 97, 256]),
    "repeat_first": dynamic(_lens({65: 1, 256: 1}, 257), [0], [], cl=_lens({16: 1, 0: 2, 1: 2}, 19), cl_seq=[16]),
    "missing_eob": dynamic(_lens({97: 1, 98: 1}, 257), [0], [97, 98]),
    "too_far": fixed_block([97, (257, 0, 0, 1, 0, 0), 256]),
    "ok_dist1": fixed_block([97, (257, 0, 0, 0, 0, 0), 256]),
    "lit286": fixed_block([97, 286, 256]),
    "lit287": fixed_block([97, 287, 256]),
    "dist30": fixed_block([97, 97, 97, (257, 0, 0, 30, 0, 0), 256]),
    "dist31": fixed_block([97, 97, 97, (257, 0, 0, 31, 0, 0), 256]),
    "no_final": fixed_block([97, 256], final=0),
    "trailing_bytes": fixed_block([97, 256]) + b"\xde\xad\xbe\xef",
}


@pytest.mark.parametrize("name", sorted(MALFORMED))
def test_malformed(ctx, name):
    _expect(ctx, MALFORMED[name])


def _expect(ctx, stream):
    from idencomp_b200 import capi
    good = zraw(b"ok\nfine", 6)
    blocks = [[good], [stream], [good]]
    if zlib_accepts(stream) is None:
        with pytest.raises(capi.IdnGpuError) as e:
            run(ctx, [slice_rec(s[0]) for s in blocks], [2, 1, 2])
        assert e.value.kind == "SerializeError" and e.value.bad_block == 1
    else:
        check(ctx, blocks, [2, 1, 2])


def test_truncation_at_every_byte(ctx):
    text = b"\n".join(bench_titles(200)) + bytes(range(256))
    stream = zraw(text[:1500], 6, flush_every=500, flush=zlib.Z_FULL_FLUSH)
    for cut in range(len(stream)):
        _expect(ctx, stream[:cut])


# ---- 5. splitting, as the host's inflate_names --------------------------------------------------------------------------
def test_splitting(ctx):
    a, b, c = zraw(b"n1\nn2\nn3"), zraw(b"x\n\ny\n"), zraw(b"")
    texts = [[a], [a], [b], [a, b], [], [c], [b, c, a], []]
    wants = [1, 5, 4, 6, 3, 2, 9, 0]
    payloads = [b"".join(slice_rec(s) for s in t) + (b"\x01\x05" if i % 2 else b"") for i, t in enumerate(texts)]
    check(ctx, texts, wants, payloads)
    got, st = run(ctx, [b"\x01\x02", b""], [3, 1])
    assert got == [b""] * 4 and st["n_streams"] == 0


def test_brotli_and_unknown_compression(ctx):
    from idencomp_b200 import capi
    good = slice_rec(zraw(b"a\nb"))
    with pytest.raises(capi.IdnGpuError) as e:
        run(ctx, [good, slice_rec(b"\x0b\x01\x80abc\x03", comp=0)], [2, 1])
    assert e.value.kind == "Unsupported"
    with pytest.raises(capi.IdnGpuError) as e:
        run(ctx, [good, good, slice_rec(zraw(b"c"), comp=2)], [2, 2, 1])
    assert e.value.kind == "SerializeError" and e.value.bad_block == 2


# ---- 6. host mirror ------------------------------------------------------------------------------------------------------
def _host_models(H, toy_models):
    return [H.Model.new(m.md.mtype, m.md.spec_name, m.md.probs, m.md.spec_keys, m.md.spec_ctx) for m in toy_models]


def _write(H, models, reads, **kw):
    c = H.IdnCompressor(models, **kw)
    c.add_batch(reads.read_off, reads.acids, reads.quals, reads.name_off, reads.names)
    idn = c.finish()
    c.close()
    return idn


def _same_reads(H, hm, idn, **kw):
    a = H.decompress(hm, idn, **kw)
    b = H.decompress(hm, idn, identifiers_on_device=True, **kw)
    for k in ("read_off", "acids", "quals", "name_off", "names"):
        assert np.array_equal(a[k], b[k]), k
    t = H.decompress_text(hm, idn)
    assert H.decompress_text(hm, idn, identifiers_on_device=True) == t
    out = np.zeros(len(t) + 64, dtype=np.uint8)
    n = H.decompress_text_into(hm, idn, out, identifiers_on_device=True)
    assert out[:n].tobytes() == t
    rd = H.FastqTextReader(hm, idn, devices=[0, 0], batch_blocks=2, identifiers_on_device=True)
    assert b"".join(v.tobytes() for v in rd) == t
    return t


@pytest.mark.parametrize("mode", [1, 2], ids=["compat", "native"])
@pytest.mark.parametrize("dev_codec", [False, True], ids=["zlib", "device_deflate"])
def test_host_mirror(toy_models, reads_1k, mode, dev_codec):
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    idn = _write(H, hm, reads_1k, max_block_total_len=3000, mode=mode, batch_blocks=4, identifiers_on_device=dev_codec)
    t = _same_reads(H, hm, idn)
    assert t == (GOLDEN / "1k-reads.fastq").read_bytes()
    _same_reads(H, hm, _write(H, hm, reads_1k, max_block_total_len=3000, mode=mode, include_identifiers=False))


def test_golden_1m(toy_models):
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    idn = (GOLDEN / "1M.idn").read_bytes()
    assert H.decompress_text(hm, idn, identifiers_on_device=True) == (GOLDEN / "1M.fastq").read_bytes()


def test_brotli_falls_back(toy_models, reads_1k):
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    try:
        idn = _write(H, hm, reads_1k, max_block_total_len=3000, quality=8)
        H.decompress(hm, idn)
    except H.HostError as e:
        if e.kind == "Unsupported":
            pytest.skip("the Brotli libraries are missing")
        raise
    _same_reads(H, hm, idn)


def _blocks(idn):
    pos = 12 + 32 * idn[11]
    out = []
    while True:
        ln = int.from_bytes(idn[pos:pos + 4], "big")
        if ln == 0:
            return idn[:12 + 32 * idn[11]], out, idn[pos:]
        out.append((idn[pos + 4:pos + 8], idn[pos + 8:pos + 8 + ln]))
        pos += 8 + ln


def test_corrupt_name_in_stored_slice(toy_models, reads_1k):
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    idn = _write(H, hm, reads_1k, max_block_total_len=3000)
    head, blocks, tail = _blocks(idn)

    def restored(corrupt):
        out = head
        for i, (crc, p) in enumerate(blocks):
            n = int.from_bytes(p[1:5], "big")
            text = zlib_accepts(p[6:6 + n])
            if i == 2 and corrupt:
                text = text[:5] + bytes([text[5] ^ 1]) + text[6:]
            p = slice_rec(zraw(text, 0)) + p[6 + n:]
            out += len(p).to_bytes(4, "big") + crc + p
        return out + tail
    _same_reads(H, hm, restored(False))
    bad = restored(True)
    for dev in (False, True):
        with pytest.raises(H.HostError) as e:
            H.decompress(hm, bad, identifiers_on_device=dev)
        assert e.value.kind == "BlockChecksumMismatch" and "block 2" in str(e.value)
        with pytest.raises(H.HostError) as e:
            H.decompress_text(hm, bad, identifiers_on_device=dev)
        assert e.value.kind == "BlockChecksumMismatch"

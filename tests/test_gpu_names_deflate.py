"""Identifiers slices Deflated on the device (csrc/idn_deflate.cuh, idn_gpu_deflate_names, IdnCompressor with
identifiers_on_device): every slice must inflate on its own with zlib to the block's names joined by '\\n', stay within the
documented bound, depend on the block's names only, and a container written this way must read back exactly as the one
written with the host's zlib."""
import random
import zlib

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

SEG = 65536  # input bytes per Deflate block of the device codec


@pytest.fixture(scope="module")
def ctx():
    from idencomp_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def _table(blocks):
    """blocks: list of lists of names (bytes) -> (name_off, names, block_first_read)"""
    names = [n for blk in blocks for n in blk]
    off = np.zeros(len(names) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(n) for n in names]) if names else []
    bf = np.zeros(len(blocks) + 1, dtype=np.uint32)
    bf[1:] = np.cumsum([len(b) for b in blocks])
    return off, np.frombuffer(b"".join(names), dtype=np.uint8), bf


def _inflate(data):
    d = zlib.decompressobj(-15)
    out = d.decompress(bytes(data))
    assert d.eof and d.unused_data == b""
    return out


def _slices(ctx, blocks):
    off, nm, bf = _table(blocks)
    out, so = ctx.deflate_names(off, nm, bf)
    bound = int(ctx.L.idn_gpu_deflate_names_bound(int(off[-1]), len(off) - 1, len(blocks)))
    assert int(so[-1]) <= bound
    res = []
    for b, blk in enumerate(blocks):
        s = out[int(so[b]):int(so[b + 1])].tobytes()
        assert s[0] == 0 and s[5] == 1 and int.from_bytes(s[1:5], "big") == len(s) - 6
        assert _inflate(s[6:]) == b"\n".join(blk), f"block {b}"
        res.append(s)
    return res


def _one(text):
    return [[text]]


def bench_titles(n, first=0):
    return [b"r%012d 1:N:0" % i for i in range(first, first + n)]


def illumina_names(n, seed=1):
    rng = random.Random(seed)
    x = y = 1000
    out = []
    for _ in range(n):
        x += rng.randint(1, 40)
        if x > 32000:
            x = 1000
            y += rng.randint(1, 300)
        out.append(b"A00123:8:H5TJ3DSXX:1:1101:%d:%d 1:N:0:ACGTACGT+TTGCAGGA" % (x, y))
    return out


def printable(n, seed=3):
    return np.random.default_rng(seed).integers(33, 127, size=n, dtype=np.uint8).tobytes()


# ---- 1. standalone call, inflated with zlib -----------------------------------------------------------------------------
def test_empty_inputs(ctx):
    _slices(ctx, [[b""]])
    _slices(ctx, [[b""] * 1000])
    _slices(ctx, [[]])
    _slices(ctx, [[b"x"]])


@pytest.mark.parametrize("n", [SEG - 1, SEG, SEG + 1, 2 * SEG + 1, 32767, 32768, 32769])
def test_lengths_around_segment_and_window(ctx, n):
    rng = np.random.default_rng(n)
    text = bytes(rng.choice(np.frombuffer(b"ACGT:0123456789", dtype=np.uint8), size=n))
    _slices(ctx, _one(text))
    _slices(ctx, _one(printable(n, seed=n)))


@pytest.mark.parametrize("dist", [32768, 32769])
def test_repeat_at_window_edge(ctx, dist):
    head = printable(512, seed=11)
    text = head + printable(dist - 512, seed=12) + head + printable(100, seed=13)
    _slices(ctx, _one(text))
    # the same as names of one block, so that the repeat spans a '\n'
    _slices(ctx, [[head, printable(dist - 513, seed=14), head]])


def test_long_runs_and_all_bytes(ctx):
    _slices(ctx, _one(b"a" * 300_000))
    _slices(ctx, [[b"a" * 1000] * 300])
    _slices(ctx, _one(bytes(range(256)) * 3))
    _slices(ctx, _one(bytes(range(256))))
    _slices(ctx, _one(np.random.default_rng(5).integers(0, 256, size=200_000, dtype=np.uint8).tobytes()))


def test_workload_shapes(ctx):
    per = 41_943
    blocks = [bench_titles(per, b * per) for b in range(24)]
    _slices(ctx, blocks)
    ill = illumina_names(per * 4)
    _slices(ctx, [ill[i * per:(i + 1) * per] for i in range(4)])


def test_one_call_from_empty_to_4mib(ctx):
    sizes = [0, 1, 100, SEG - 1, SEG, 3 * SEG + 7, 1 << 20, 4 << 20]
    rng = random.Random(9)
    blocks = []
    for s in sizes:
        names, n = [], 0
        while n < s:
            k = min(rng.randint(1, 300), s - n)
            names.append(bytes(rng.choice(b"ACGT:_0123456789") for _ in range(k)) if k < 40 else printable(k, seed=n))
            n += k + 1
        blocks.append(names if s else [])
    _slices(ctx, blocks)


def test_incompressible_names_stay_within_the_bound(ctx):
    rng = np.random.default_rng(17)
    for n_reads, ln in ((1, 3 * SEG), (5000, 37), (20000, 1)):
        names = [rng.integers(0, 256, size=ln, dtype=np.uint8).tobytes() for _ in range(n_reads)]
        _slices(ctx, [names[: n_reads // 2], names[n_reads // 2:]])


# ---- 2. ratio against zlib level 6 -------------------------------------------------------------------------------------
def _zlib6(blocks):
    total = 0
    for blk in blocks:
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        total += len(c.compress(b"\n".join(blk)) + c.flush())
    return total


@pytest.mark.parametrize("shape,bar", [("bench", 1.05), ("illumina", 1.25), ("printable", 1.05)])
def test_ratio_against_zlib6(ctx, shape, bar):
    per = 41_943
    if shape == "bench":
        blocks = [bench_titles(per, b * per) for b in range(4)]
    elif shape == "illumina":
        ill = illumina_names(per * 4)
        blocks = [ill[i * per:(i + 1) * per] for i in range(4)]
    else:
        blocks = [[printable(19 * per, seed=b)] for b in range(4)]
    got = sum(len(s) - 6 for s in _slices(ctx, blocks))
    want = _zlib6(blocks)
    assert got <= bar * want, f"{shape}: device {got} bytes, zlib-6 {want} bytes ({got / want:.3f})"


# ---- 3. determinism ----------------------------------------------------------------------------------------------------
def test_slices_depend_only_on_their_block(ctx):
    rng = random.Random(21)
    ill = illumina_names(16 * 3000, seed=5)
    blocks = [ill[i * 3000:(i + 1) * 3000] if i % 3 else bench_titles(rng.randint(0, 9000), i * 10_000) for i in range(16)]
    all1 = _slices(ctx, blocks)
    assert _slices(ctx, blocks) == all1
    assert [_slices(ctx, [blk])[0] for blk in blocks] == all1
    order = list(range(16))
    rng.shuffle(order)
    shuffled = _slices(ctx, [blocks[i] for i in order])
    assert [shuffled[order.index(i)] for i in range(16)] == all1


# ---- 4. host mirror ----------------------------------------------------------------------------------------------------
def _host_models(H, toy_models):
    return [H.Model.new(m.md.mtype, m.md.spec_name, m.md.probs, m.md.spec_keys, m.md.spec_ctx) for m in toy_models]


def _blocks(idn):
    """container -> list of (crc, payload) of its blocks"""
    pos = 12 + 32 * idn[11]
    out = []
    while True:
        ln = int.from_bytes(idn[pos:pos + 4], "big")
        if ln == 0:
            return out
        out.append((idn[pos + 4:pos + 8], idn[pos + 8:pos + 8 + ln]))
        pos += 8 + ln


def _split_ids(payload):
    assert payload[0] == 0 and payload[5] == 1
    n = int.from_bytes(payload[1:5], "big")
    return _inflate(payload[6:6 + n]), payload[6 + n:]


def _write(H, models, reads, how, text=None, **kw):
    c = H.IdnCompressor(models, **kw)
    if how == "batch":
        c.add_batch(reads.read_off, reads.acids, reads.quals, reads.name_off, reads.names)
    elif how == "sequence":
        for r in range(reads.n_reads):
            a, b = int(reads.read_off[r]), int(reads.read_off[r + 1])
            c.add_sequence(reads.name(r), reads.acids[a:b], reads.quals[a:b])
    else:
        c.add_fastq_text(text)
    idn = c.finish()
    st = c.stats()
    c.close()
    return idn, st


@pytest.mark.parametrize("mode", [1, 2], ids=["compat", "native"])
def test_host_mirror_device_names(O, toy_models, reads_1k, mode):
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    text = (GOLDEN / "1k-reads.fastq").read_bytes()
    kw = dict(max_block_total_len=3000, mode=mode, batch_blocks=4, text=text)
    ref, ref_st = _write(H, hm, reads_1k, "batch", **kw)
    dev = {how: _write(H, hm, reads_1k, how, identifiers_on_device=True, **kw) for how in ("batch", "sequence", "text")}
    assert dev["batch"][0] == dev["sequence"][0] == dev["text"][0]
    idn, st = dev["batch"]
    rb, db = _blocks(ref), _blocks(idn)
    assert len(rb) == len(db) > 1
    ids_bytes = 0
    for (rc, rp), (dc, dp) in zip(rb, db):
        assert rc == dc
        rn, rrest = _split_ids(rp)
        dn, drest = _split_ids(dp)
        assert rn == dn and rrest == drest
        ids_bytes += len(dp) - len(drest)
    assert st["out_identifier_bytes"] == ids_bytes and dev["text"][1]["out_identifier_bytes"] == ids_bytes
    assert st["out_payload_bytes"] == ref_st["out_payload_bytes"]
    a, b = H.decompress(hm, ref), H.decompress(hm, idn)
    for k in ("read_off", "acids", "quals", "name_off", "names"):
        assert np.array_equal(a[k], b[k]), k
    ta = b"".join(v.tobytes() for v in H.FastqTextReader(hm, ref))
    tb = b"".join(v.tobytes() for v in H.FastqTextReader(hm, idn))
    assert ta == tb == text
    # two contexts on one device give the same file
    assert _write(H, hm, reads_1k, "batch", identifiers_on_device=True, devices=[0, 0], **kw)[0] == idn
    # without identifiers the flag changes nothing
    off = dict(kw, include_identifiers=False)
    assert _write(H, hm, reads_1k, "batch", identifiers_on_device=True, **off)[0] == _write(H, hm, reads_1k, "batch", **off)[0]


def test_golden_1m_names(O, toy_models, reads_1m):
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    text = (GOLDEN / "1M.fastq").read_bytes()
    for how in ("batch", "text"):
        idn, _ = _write(H, hm, reads_1m, how, text=text, identifiers_on_device=True)
        (crc, payload), = _blocks(idn)
        names, _ = _split_ids(payload)
        assert names == b"data/SRR1518133_1.fastq 0:500000"
        d = H.decompress(hm, idn)
        assert np.array_equal(d["acids"], reads_1m.acids) and np.array_equal(d["quals"], reads_1m.quals)


# ---- 5. errors ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("quality", [8, 9])
def test_brotli_qualities_are_unsupported(toy_models, quality):
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    with pytest.raises(H.HostError) as e:
        H.IdnCompressor(hm, quality=quality, identifiers_on_device=True)
    assert e.value.kind == "Unsupported"
    H.IdnCompressor(hm, quality=quality, identifiers_on_device=True, include_identifiers=False).close()


def test_bad_tables_and_small_output(ctx):
    from idencomp_b200 import capi
    off, nm, bf = _table([bench_titles(100), bench_titles(50)])
    bad_off = off.copy()
    bad_off[10] = bad_off[9] - 1
    with pytest.raises(capi.IdnGpuError) as e:
        ctx.deflate_names(bad_off, nm, bf)
    assert e.value.kind == "InvalidArgument"
    for bad_bf in ([0, 120, 100, 150], [1, 100, 150]):
        with pytest.raises(capi.IdnGpuError) as e:
            ctx.deflate_names(off, nm, np.array(bad_bf, dtype=np.uint32))
        assert e.value.kind == "InvalidArgument"
    _, so = ctx.deflate_names(off, nm, bf)
    need = int(so[-1])
    with pytest.raises(capi.IdnGpuError) as e:
        ctx.deflate_names(off, nm, bf, out_cap=need - 1)
    assert e.value.kind == "NoSpace" and e.value.required == need
    out, so2 = ctx.deflate_names(off, nm, bf, out_cap=need)
    assert np.array_equal(so, so2) and len(out) == need

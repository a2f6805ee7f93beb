"""The device FASTQ reader (csrc/idn_fastq.cuh) against the oracle's sequential statement of FastqReader::read_sequence
(fastq/reader.rs:166-282): which error is reported and for which record, ASCII white space, the newline tiles and the
line-state scan tiles, the chunked entry point idn_gpu_fastq_parse_chunk and the host mirror's add_fastq_text.

Every device result is compared with the oracle on the same input: read_off, acids, quals, name_off and names, or, for
rejected input, the FastqReaderError variant and the 0-based record in file order.  The oracle-only tests are unmarked so
that they run without a GPU."""
import ctypes as C
import re

import numpy as np
import pytest

from conftest import GOLDEN

WS = b"\t\n\x0b\x0c\r "  # ASCII white space: bytes 9-13 and 32, what str::trim strips of ASCII
WS_IN_LINE = WS.replace(b"\n", b"")

# ---------------------------------------------------------------------------------------------------------------------
# the hand table
# ---------------------------------------------------------------------------------------------------------------------
# One defect per entry, in the order the reference checks a record: the title starts with '@', the acids line is there,
# every acid is valid, the separator line is there and starts with '+', the quality line is there, every quality byte
# of the whole line is valid, the two lengths are equal.  (overrides of _rec(), line the defect sits on, variant)
DEFECTS = {
    "title": (dict(title=b"r"), 0, "InvalidFormat"),
    "eof_acids": (dict(lines=1), 1, "EofReached"),
    "acid": (dict(acids=b"AXGT"), 1, "InvalidAcid"),
    "eof_sep": (dict(lines=2), 2, "EofReached"),
    "sep": (dict(sep=b"-"), 2, "InvalidFormat"),
    "eof_qual": (dict(lines=3), 3, "EofReached"),
    "qual": (dict(qual=b"II I"), 3, "InvalidQualityScore"),
    "length": (dict(qual=b"III"), 3, "AcidAndQualityScoreLengthMismatch"),
}
EOF_DEFECTS = ("eof_acids", "eof_sep", "eof_qual")


def _rec(title=b"@r", acids=b"ACGT", sep=b"+", qual=b"IIII", lines=4):
    return b"".join(line + b"\n" for line in (title, acids, sep, qual)[:lines])


def _defective(names, title=b"@r"):
    """one record holding every defect in `names`, and the variant the reference stops at"""
    kw = dict(title=title)
    for d in names:
        kw.update(DEFECTS[d][0])
    if "qual" in names and "length" in names:
        kw["qual"] = b"I I"  # a bad byte and a short line: the bytes are checked first
    kw["lines"] = min([DEFECTS[d][0]["lines"] for d in names if d in EOF_DEFECTS] + [4])
    reached = [d for d in DEFECTS if d in names and (DEFECTS[d][1] < kw["lines"] or DEFECTS[d][0].get("lines") == kw["lines"])]
    return _rec(**kw), DEFECTS[reached[0]][2]


def _hand_table():
    """(id, text, expected): expected = (variant, record) for rejected input, the list of titles for accepted input"""
    good = _rec(b"@ok")
    cases = [
        # the first error in file order, whatever kind the later one is
        ("issue_acid_then_title", b"@a\nAXGT\n+\n!!!!\nr2\nAC\n+\n!!\n", ("InvalidAcid", 0)),
        ("issue_cut_after_bad_acids", b"@a\nAXGT\n", ("InvalidAcid", 0)),
        ("issue_cut_after_bad_separator", b"@a\nACGT\n-\n", ("InvalidFormat", 0)),
        ("long_quality_line_bad_byte", _rec(qual=b"IIII I"), ("InvalidQualityScore", 0)),
        ("crlf_quality", b"@a\nACGT\n+\nIIII\r\n", ("InvalidQualityScore", 0)),
        ("empty_separator", b"@a\nA\n\nI\n", ("InvalidFormat", 0)),
        ("cut_inside_first_line", b"@a", ("EofReached", 0)),
        ("cut_acids_without_newline", b"@a\nAC", ("EofReached", 0)),
    ]
    for d in DEFECTS:
        text, kind = _defective([d])
        cases.append((f"one_{d}", good + text, (kind, 1)))
    names = list(DEFECTS)
    for i, x in enumerate(names):
        for y in names[i + 1:]:
            text, kind = _defective([x, y])
            cases.append((f"same_record_{x}+{y}", good + text, (kind, 1)))
    for x in names:
        if x in EOF_DEFECTS:
            continue  # only the last record can end early
        for y in names:
            if y != x:
                cases.append((f"records_{x}_then_{y}", good + _defective([x])[0] + _defective([y])[0], (DEFECTS[x][2], 1)))
    for c in WS:
        w = bytes([c])
        cases += [
            (f"blank_lines_{c}", w + b"\n" + w * 3 + b"\n" + _rec(b"@a") + w + b"\n\n" + _rec(b"@b") + w, [b"a", b"b"]),
            (f"blank_line_before_title_only_{c}", w + b"\n" + _rec(b"@a"), [b"a"]),
        ]
    for c in WS_IN_LINE:
        w = bytes([c])
        cases += [
            (f"title_ends_{c}", _rec(b"@" + w + b"a" + w) + _rec(b"@" + w * 2 + b"b c" + w * 2), [b"a", b"b c"]),
            (f"title_inside_{c}", _rec(b"@a" + w + b"b"), [b"a" + w + b"b"]),
            (f"title_only_white_space_{c}", _rec(b"@" + w), [b""]),
            (f"white_space_before_at_{c}", good + _rec(w + b"@a"), ("InvalidFormat", 1)),
            (f"white_space_acids_line_{c}", _rec(acids=w, qual=b"I"), ("InvalidAcid", 0)),
            (f"white_space_separator_{c}", _rec(sep=w), ("InvalidFormat", 0)),
            (f"white_space_quality_{c}", _rec(acids=b"A", qual=w), ("InvalidQualityScore", 0)),
            (f"last_line_white_space_no_newline_{c}", _rec(b"@a") + w * 2, [b"a"]),
        ]
    cases += [
        ("issue_lone_vt_line", b"\x0b\n@a\nA\n+\n!\n", [b"a"]),
        ("issue_title_ends_ff", b"@ a\x0c\nA\n+\n!\n", [b"a"]),
        ("zero_length_read", b"@e\n\n+\n\n" + good, [b"e", b"ok"]),
        ("zero_length_read_cut_before_quality", b"@e\n\n+\n", ("EofReached", 0)),
        ("at_alone", b"@\nA\n+\n!", [b""]),
    ]
    return cases


HAND = _hand_table()


def _oracle(O, text):
    try:
        return O.fastq_parse(text)
    except O.OracleError as e:
        assert hasattr(e, "fastq_error"), str(e)
        return e.fastq_error, e.bad_record


@pytest.mark.parametrize("text,expected", [c[1:] for c in HAND], ids=[c[0] for c in HAND])
def test_oracle_hand_table(O, text, expected):
    got = _oracle(O, text)
    if isinstance(expected, tuple):
        assert got == expected
    else:
        assert not isinstance(got, tuple), got
        assert [got.name(r) for r in range(got.n_reads)] == expected


def test_oracle_error_names_match_capi(O):
    from idencomp_b200 import capi
    kinds = {k for _, _, e in HAND if isinstance(e, tuple) for k in [e[0]]}
    assert kinds == set(capi.FASTQ_ERRORS.values())


# ---------------------------------------------------------------------------------------------------------------------
# device helpers
# ---------------------------------------------------------------------------------------------------------------------
FIELDS = ("read_off", "acids", "quals", "name_off", "names")


@pytest.fixture(scope="module")
def gctx():
    from idencomp_b200 import capi
    ctx = capi.Context(0)
    yield ctx
    ctx.close()


def _device(gctx, text):
    from idencomp_b200.capi import IdnGpuError
    try:
        return gctx.fastq_parse(text)
    except IdnGpuError as e:
        assert e.kind == "SerializeError", str(e)
        return e.fastq_error, e.bad_record


def agree(gctx, O, text, what=""):
    """the device and the oracle give the same arrays, or reject the text with the same (variant, record)"""
    want, got = _oracle(O, text), _device(gctx, text)
    if isinstance(want, tuple):
        assert len(got) == 2, f"{what}: the device accepts, the oracle says {want}"
        assert got == want, f"{what}: device {got}, oracle {want}"
    else:
        assert len(got) == 5, f"{what}: the device says {got}, the oracle accepts"
        ref = (want.read_off, want.acids, want.quals, want.name_off, want.names)
        for f, x, y in zip(FIELDS, got, ref):
            assert np.array_equal(x, y), f"{what}: {f} differs"
    return want, got


def dirty_text(rng, n_records, *, long_reads=0, max_len=60, final_newline=None):
    """A valid FASTQ text in the forms the reader must accept: blank and white-space-only lines (every ASCII white-space
    byte, a lone '\\r', a lone '\\x0b') before titles, titles with white space at both ends, empty titles and '@' alone,
    '+title' separators, zero-length reads, `long_reads` reads of 64 KiB or more, a final newline or none.
    -> (text, title_off, rec_end, title_line): byte offset of every title line and of the end of every record, and the
    line number of every title."""
    parts, title_off, rec_end, title_line = [], [], [], []
    pos = line = 0
    long_at = set(rng.choice(n_records, size=long_reads, replace=False).tolist()) if long_reads else set()

    def ws(k):
        return bytes(rng.choice(np.frombuffer(WS_IN_LINE, dtype=np.uint8), size=k))

    def put(b, lines):
        nonlocal pos, line
        parts.append(b)
        pos += len(b)
        line += lines

    for r in range(n_records):
        if rng.random() < 0.3:
            for _ in range(int(rng.integers(1, 4))):
                blank = [b"", b"\r", b"\x0b", ws(int(rng.integers(1, 6)))][int(rng.integers(0, 4))]
                put(blank + b"\n", 1)
        u = rng.random()
        if u < 0.05:
            name = b""
        elif u < 0.1:
            name = ws(int(rng.integers(1, 3)))
        else:
            name = bytes(rng.integers(33, 127, size=int(rng.integers(1, 20)), dtype=np.uint8))
            if rng.random() < 0.3:
                name += b" " + bytes(rng.integers(33, 127, size=int(rng.integers(1, 8)), dtype=np.uint8))
            if rng.random() < 0.3:
                name = ws(int(rng.integers(1, 3))) + name + ws(int(rng.integers(0, 3)))
        if r in long_at:
            ln = (1 << 16) + int(rng.integers(0, 9000))
        elif rng.random() < 0.1:
            ln = 0
        else:
            ln = int(rng.integers(1, max_len + 1))
        acids = bytes(rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), size=ln))
        quals = bytes(rng.integers(33, 127, size=ln, dtype=np.uint8))
        sep = b"+" + (name if rng.random() < 0.3 else b"")
        title_off.append(pos)
        title_line.append(line)
        put(b"@" + name + b"\n" + acids + b"\n" + sep + b"\n" + quals + b"\n", 4)
        rec_end.append(pos)
    if rng.random() < 0.3:
        put(ws(int(rng.integers(1, 4))) + b"\n", 1)
    text = b"".join(parts)
    if final_newline is None:
        final_newline = rng.random() < 0.5
    if not final_newline and len(text) >= 2 and text[-2:-1] != b"\n":  # an empty last line would vanish with its newline
        text = text[:-1]
        rec_end = [min(e, len(text)) for e in rec_end]
    return text, np.asarray(title_off), np.asarray(rec_end), np.asarray(title_line)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the hand table, dirty texts, tile edges, scale, mutations
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("text,expected", [c[1:] for c in HAND], ids=[c[0] for c in HAND])
def test_device_hand_table(gctx, O, text, expected):
    want, got = agree(gctx, O, text)
    if isinstance(expected, tuple):
        assert got == expected
    else:
        ro, a, q, no, nm = got
        assert [nm[no[r]:no[r + 1]].tobytes() for r in range(len(ro) - 1)] == expected


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(6))
def test_dirty_texts_and_round_trip(gctx, O, seed):
    rng = np.random.default_rng(100 + seed)
    text, *_ = dirty_text(rng, 400, long_reads=2 if seed < 3 else 0)
    want, got = agree(gctx, O, text, f"seed {seed}")
    assert not isinstance(want, tuple), want
    # FastqWriter over the device's parse == the oracle's writer over its own
    assert gctx.fastq_format(*got) == O.fastq_write(want)


def _pad_to_newline(prefix, p, role):
    """prefix + one more line whose '\\n' lands on byte p: a blank line of spaces, or the title, acids or quality line of
    a record"""
    room = p - len(prefix)
    if role == "blank":
        out = prefix + b" " * room + b"\n"
    elif role == "title":
        out = prefix + b"@" + b"t" * (room - 1) + b"\n"
    elif role == "acids":
        out = prefix + b"@t\n" + b"A" * (room - 3) + b"\n"
    else:  # quality line of a 40-symbol read
        k = room - 2 * 40 - 5
        out = prefix + b"@" + b"t" * k + b"\n" + b"C" * 40 + b"\n+\n" + b"#" * 40 + b"\n"
    assert out[p] == ord("\n") and len(out) == p + 1
    if role == "title":
        out += b"A\n+\n#\n"
    elif role == "acids":
        out += b"+\n" + b"#" * (room - 3) + b"\n"
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("p", [4095, 4096, 4097, 8191, 8192, 8193])
@pytest.mark.parametrize("role", ["blank", "title", "acids", "quality"])
def test_newline_at_newline_tile_edges(gctx, O, p, role):
    """kFqTile = 4096 bytes per block of the newline count / scatter passes"""
    rng = np.random.default_rng(p)
    prefix, title_off, *_ = dirty_text(rng, 200, max_len=30, final_newline=True)
    prefix = prefix[:title_off[title_off < p - 200][-1]]
    text = _pad_to_newline(prefix, p, role)
    tail, *_ = dirty_text(rng, 5, final_newline=True)
    agree(gctx, O, text, f"{role} newline at {p}, text ends there")
    want, _ = agree(gctx, O, text + tail, f"{role} newline at {p}")
    assert not isinstance(want, tuple), want
    agree(gctx, O, text + tail[:-1], f"{role} newline at {p}, no final newline")


@pytest.mark.gpu
def test_last_byte_of_text_on_tile_edges(gctx, O):
    rng = np.random.default_rng(5)
    base, *_ = dirty_text(rng, 300, max_len=30, final_newline=True)
    for n in (4095, 4096, 4097, 8192):
        text = base[:n]
        cut = text.rfind(b"\n") + 1
        # the text ends with its '\n' at byte n - 1, or with an unterminated line there
        blank_end = text[:cut] + b" " * max(0, n - cut - 1) + b"\n"
        agree(gctx, O, blank_end[:n], f"ends at {n}")
        agree(gctx, O, text, f"cut at {n}")


def _records_at_lines(rng, targets, defect_at=None):
    """records whose titles sit on the given line numbers, blank lines as padding; a bad acid in the record whose title
    is on line defect_at"""
    lines, tl = [], []
    for t in targets:
        while len(lines) + 4 + 1 <= t:
            ln = int(rng.integers(0, 12))
            lines += [b"@p", b"A" * ln, b"+", b"!" * ln]
        while len(lines) < t:
            lines.append(b"" if rng.random() < 0.5 else b" \t")
        ac = b"ACXGT" if t == defect_at else b"ACGT"
        tl.append(len(lines))
        lines += [b"@t%d" % t, ac, b"+", b"I" * len(ac)]
    return b"\n".join(lines) + b"\n", tl


@pytest.mark.gpu
def test_records_at_scan_tile_edges(gctx, O):
    """kFstTile = 2048 lines per tile of the line-state scan, 8 lines per thread"""
    for targets in ([7, 2047, 4096, 6145], [8, 2048, 4097, 6143], [9, 2049, 4095, 6144]):
        text, tl = _records_at_lines(np.random.default_rng(targets[0]), targets)
        assert tl == targets
        agree(gctx, O, text, f"titles on lines {targets}")
        for t in targets[1:]:
            text, _ = _records_at_lines(np.random.default_rng(targets[0]), targets, defect_at=t)
            want, _ = agree(gctx, O, text, f"bad acid in the record on line {t}")
            assert want[0] == "InvalidAcid"


@pytest.mark.gpu
def test_more_scan_tiles_than_threads(gctx, O):
    """more than 256 x 2048 lines: every thread of fst_tiles_kernel chains more than one tile"""
    rng = np.random.default_rng(11)
    n = 165_000
    lens = rng.integers(0, 20, size=n)
    blanks = rng.integers(0, 3, size=n) * (rng.random(n) < 0.12)
    acgt = np.frombuffer(b"ACGTN", dtype=np.uint8)
    pool_a = bytes(rng.choice(acgt, size=64))
    pool_q = bytes(rng.integers(33, 127, size=64, dtype=np.uint8))
    parts, title_line, title_off = [], [], []
    line = pos = 0
    for r in range(n):
        pad = b"\n" * int(blanks[r])
        ln = int(lens[r])
        s = int(rng.integers(0, 32)) if r % 7 == 0 else 0
        rec = b"@r%d\n%s\n+\n%s\n" % (r, pool_a[s:s + ln], pool_q[s:s + ln])
        title_off.append(pos + len(pad))
        title_line.append(line + int(blanks[r]))
        parts += [pad, rec]
        pos += len(pad) + len(rec)
        line += int(blanks[r]) + 4
    text = b"".join(parts)
    assert line > 600_000
    # records straddle the 2048-line scan tiles at every phase
    title_line = np.asarray(title_line)
    edges = np.arange(2048, line, 2048)
    owner = np.searchsorted(title_line, edges, side="right") - 1
    phase = edges - title_line[owner]
    assert set(phase[phase < 4].tolist()) == {0, 1, 2, 3}
    agree(gctx, O, text, "valid")
    # a bad acid deep in the text, and a title without '@' after it
    k = int(np.nonzero(lens[140_000:] > 0)[0][0]) + 140_000
    a = title_off[k] + len(b"@r%d\n" % k)
    t2 = title_off[k + 1000]
    bad = bytearray(text)
    bad[a] = ord("X")
    bad[t2] = ord("r")
    want, got = agree(gctx, O, bytes(bad), "deep defects")
    assert got == ("InvalidAcid", k)


def _mutate(rng, text):
    t = bytearray(text)
    kind = int(rng.integers(0, 5))
    i = int(rng.integers(0, len(t)))
    if kind == 0:
        t[i] = int(rng.integers(0, 256))
    elif kind == 1:
        t[i] = b"@+\n \r\x0b"[int(rng.integers(0, 6))]
    elif kind == 2:
        del t[i]
    elif kind == 3:
        t.insert(i, ord("\n"))
    else:
        nl = [j for j, c in enumerate(t) if c == 10]
        del t[nl[int(rng.integers(0, len(nl)))]]
    return bytes(t)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_mutation_sweep(gctx, O, seed):
    rng = np.random.default_rng(200 + seed)
    text, *_ = dirty_text(rng, 150, max_len=40)
    assert not isinstance(_oracle(O, text), tuple)
    outcomes = set()
    for e in range(300):
        m = _mutate(rng, text)
        want, _ = agree(gctx, O, m, f"seed {seed} edit {e}")
        outcomes.add(want[0] if isinstance(want, tuple) else "ok")
    assert len(outcomes) >= 5, outcomes  # the edits reach most of the variants


@pytest.mark.gpu
def test_every_truncation(gctx, O):
    rng = np.random.default_rng(300)
    text, *_ = dirty_text(rng, 40, max_len=30, final_newline=True)
    text = text[:2000]
    for n in range(len(text) + 1):
        agree(gctx, O, text[:n], f"first {n} bytes")


# ---------------------------------------------------------------------------------------------------------------------
# GPU: idn_gpu_fastq_parse_chunk
# ---------------------------------------------------------------------------------------------------------------------
def _parse_chunk(gctx, text, final, max_len):
    from idencomp_b200 import capi
    ck = capi.FastqChunk()
    buf = np.frombuffer(text, dtype=np.uint8)
    rc = gctx.L.idn_gpu_fastq_parse_chunk(gctx.h, buf.ctypes.data if buf.size else None, buf.size, final, max_len, C.byref(ck))
    return rc, ck


def _chunk_blocks(gctx, ck):
    bf = np.zeros(ck.n_blocks + 1, dtype=np.uint32)
    gctx.check(gctx.L.idn_gpu_fastq_chunk_fetch(gctx.h, None, None, bf.ctypes.data, None, None, None))
    return bf


@pytest.mark.gpu
def test_parse_chunk_at_every_line_boundary(gctx, O):
    from gpu_util import blocks_of
    from idencomp_b200 import capi
    rng = np.random.default_rng(400)
    max_len = 101
    text, title_off, rec_end, _ = dirty_text(rng, 60, max_len=40, final_newline=True)
    reads = O.fastq_parse(text)
    whole = blocks_of(reads, max_len)
    cuts = [0] + [i + 1 for i, c in enumerate(text) if c == ord("\n")]
    for cut in cuts:
        rc, ck = _parse_chunk(gctx, text[:cut], 0, max_len)
        assert rc == 0, f"cut {cut}: {gctx.L.idn_gpu_last_error(gctx.h).decode()}"
        # the rule: the record cut short at the end stays, blocks form over the complete ones, and the last block stays
        # with its text for the next call
        complete = int(np.sum(rec_end <= cut))
        cut_short = complete < len(title_off) and title_off[complete] < cut
        if complete == 0:
            n_reads, n_blocks, consumed = 0, 0, int(title_off[0]) if cut_short else cut
        else:
            bf = blocks_of(O.Reads(reads.read_off[:complete + 1], reads.acids, reads.quals), max_len)
            n_blocks = len(bf) - 2
            n_reads = int(bf[-2])
            consumed = int(title_off[n_reads])
        assert (ck.n_reads, ck.n_blocks, ck.consumed_text) == (n_reads, n_blocks, consumed), f"cut {cut}"
        assert ck.n_symbols == reads.read_off[n_reads] and ck.n_name_bytes == reads.name_off[n_reads]
        first = _chunk_blocks(gctx, ck)[:n_blocks]
        rc, ck2 = _parse_chunk(gctx, text[consumed:], 1, max_len)
        assert rc == 0
        assert n_reads + ck2.n_reads == reads.n_reads and consumed + ck2.consumed_text == len(text)
        rest = _chunk_blocks(gctx, ck2).astype(np.int64) + n_reads
        assert np.array_equal(np.concatenate([first, rest]), whole), f"cut {cut}"
    # a piece of a longer input must end on a line boundary once it holds a record
    for cut in range(int(title_off[0]) + 1, int(rec_end[3])):
        if text[cut - 1] != ord("\n"):
            rc, _ = _parse_chunk(gctx, text[:cut], 0, max_len)
            assert capi.ERRORS.get(rc) == "InvalidArgument", f"cut {cut}"


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the host mirror (IdnCompressor::add_fastq_text)
# ---------------------------------------------------------------------------------------------------------------------
def _host_models(H, toy_models):
    return [H.Model.new(m.md.mtype, m.md.spec_name, m.md.probs, m.md.spec_keys, m.md.spec_ctx) for m in toy_models]


def _by_batch(H, models, reads, **kw):
    c = H.IdnCompressor(models, **kw)
    try:
        names = kw.get("include_identifiers", True)
        c.add_batch(reads.read_off, reads.acids, reads.quals, reads.name_off if names else None, reads.names if names else None)
        return c.finish()
    finally:
        c.close()


def _by_text(H, models, text, cuts, **kw):
    c = H.IdnCompressor(models, **kw)
    try:
        pos = 0
        for cut in list(cuts) + [len(text)]:
            c.add_fastq_text(text[pos:cut])
            pos = cut
        return c.finish()
    finally:
        c.close()


@pytest.fixture(scope="module")
def small_dirty(O):
    text, title_off, *_ = dirty_text(np.random.default_rng(500), 40, max_len=40)
    text = text[:title_off[title_off < 1500][-1]] + b"@end\nACGT\n+\nIIII"
    return text, O.fastq_parse(text)


@pytest.mark.gpu
def test_host_text_two_pieces_at_every_offset(O, toy_models, small_dirty):
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    text, reads = small_dirty
    kw = dict(max_block_total_len=150, mode=1, include_identifiers=True, text_chunk_bytes=64, batch_blocks=2)
    want = _by_batch(H, hm, reads, **kw)
    for cut in range(len(text) + 1):
        assert _by_text(H, hm, text, [cut], **kw) == want, f"cut {cut}"


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1, 64, 700])
@pytest.mark.parametrize("mode", [1, 2], ids=["compat", "native"])
@pytest.mark.parametrize("names", [True, False], ids=["names", "no_names"])
def test_host_text_chunk_sizes(O, toy_models, small_dirty, chunk, mode, names):
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    text, reads = small_dirty
    kw = dict(max_block_total_len=150, mode=mode, include_identifiers=names, text_chunk_bytes=chunk, batch_blocks=2)
    want = _by_batch(H, hm, reads, **kw)
    if mode == 1 and not names:
        assert want == O.compress(toy_models, reads, max_block_total_len=150, include_identifiers=False)
    rng = np.random.default_rng(chunk * 4 + mode * 2 + names)
    for k in (0, 1, 3, 12):
        cuts = sorted(rng.integers(0, len(text) + 1, size=k).tolist())
        assert _by_text(H, hm, text, cuts, **kw) == want, f"cuts {cuts}"
        assert _by_text(H, hm, text, cuts, devices=[0, 0], **kw) == want, f"two workers, cuts {cuts}"


@pytest.mark.gpu
def test_block_size_limits(O, toy_models):
    """an odd max_block_total_len: a read of max_len // 2 is the longest accepted (idn/compressor.rs:542-544), and a read
    that would push a block past max_len opens the next one (:526-540)"""
    from gpu_util import blocks_of
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    max_len = 101

    def text_of(lengths):
        rng = np.random.default_rng(sum(lengths))
        out = []
        for i, ln in enumerate(lengths):
            out.append(b"@b%d\n%s\n+\n%s\n" % (i, bytes(rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), size=ln)),
                                               bytes(rng.integers(33, 127, size=ln, dtype=np.uint8))))
        return b"".join(out)

    # blocks of exactly max_len (one with a zero-length read at its end) and reads that would make max_len + 1
    lengths = [50, 50, 1, 50, 50, 2, 49, 50, 0, 50, 50, 1, 0, 7]
    text = text_of(lengths)
    reads = O.fastq_parse(text)
    assert blocks_of(reads, max_len).tolist() == [0, 3, 5, 9, 13, 14]
    want = O.compress(toy_models, reads, max_block_total_len=max_len, include_identifiers=False)
    kw = dict(max_block_total_len=max_len, mode=1, include_identifiers=False)
    assert _by_batch(H, hm, reads, **kw) == want
    for chunk in (1, 40, 1 << 20):
        assert _by_text(H, hm, text, [], text_chunk_bytes=chunk, **kw) == want, f"chunk {chunk}"
    # the longest read accepted, and one symbol more
    for ln, ok in ((max_len // 2, True), (max_len // 2 + 1, False)):
        text = text_of([3, ln, 3])
        reads = O.fastq_parse(text)
        if ok:
            assert _by_text(H, hm, text, [], **kw) == _by_batch(H, hm, reads, **kw)
            continue
        for f in (lambda: _by_text(H, hm, text, [], **kw), lambda: _by_batch(H, hm, reads, **kw)):
            with pytest.raises(H.HostError) as e:
                f()
            assert e.value.code == 4, str(e.value)


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, [0, 0]], ids=["one_worker", "two_workers"])
def test_host_error_names_the_file_record(toy_models, devices):
    """the record is counted from the start of the input, not from the start of the chunk it was found in"""
    from idencomp_b200 import host as H
    hm = _host_models(H, toy_models)
    text = (GOLDEN / "1k-reads.fastq").read_bytes()
    lines = text.split(b"\n")
    bad_line = 4 * 777 + 1
    at = len(b"\n".join(lines[:bad_line])) + 1 + 5
    assert at > 9000  # not in the first chunk: earlier chunks are consumed before the bad one is parsed
    bad = text[:at] + b"X" + text[at + 1:]
    c = H.IdnCompressor(hm, max_block_total_len=3000, text_chunk_bytes=9000, devices=devices)
    with pytest.raises(H.HostError) as e:
        c.add_fastq_text(bad)
        c.finish()
    c.close()
    m = re.search(r"FastqReaderError::(\w+) at record (\d+)", str(e.value))
    assert m and (m.group(1), int(m.group(2))) == ("InvalidAcid", 777), str(e.value)

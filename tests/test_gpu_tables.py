"""The codec tables against the CPU oracle with adversarial frequency rows, on every table path; the per-read decoder.

Models built from data reach the branches of the table lookups only by chance: a bundled row rarely holds a frequency-1
symbol where a search branches, and uniformly random reads mostly land on the dummy row.  Here every context row is
built on purpose.  An integer frequency vector f (each >= 1, sum 2^14) leaves the quantiser unchanged when it is given
as probs = f / 16384 in f32 (every partial sum is an exact f32 integer), so the oracle and the device see exactly the
rows below:

* q-score rows (94 symbols): one dominant symbol at 0, 47 or 93 (the last puts 92 starts into bucket 0 and needs 22
  window advances of q_find); near-uniform rows; starts on every multiple of 128 and one slot to either side;
  exactly 3 .. 8 starts inside one 128-slot bucket behind owners at every offset mod 4 (the advance threshold of q_find
  and the j = 5 / 6 edge of q_find_win); powers of two and 2^k +- 1 (the encoder's reciprocal shift); two dominant
  symbols among frequency-1 runs; a Dirichlet row with a tiny alpha;
* acid rows (5 symbols): each symbol at 16 380 beside frequency-1 symbols, adjacent boundaries, powers of two,
  near-uniform.

A CPU restatement of the row layouts of idn_device.cuh (bucket LUT, windows of 4g .. 4g+7, window rows {s0, starts of
s0 .. s0+6}) runs over all 16 384 slots of every row and asserts that the set reaches every branch.  On the GPU the
rows serve as the contexts of acid and q-score models, mapped onto the spec space by a multiplicative hash with about
one spec in eight left to the dummy row, for each specialised kernel pair SP0-SP7, a run-time-generic dense pair with
position bits, a dense acid spec space too large for the per-spec acid tables (adirect / aenc) and a hashed pair.
Uniformly random reads code every (row, symbol) pair (counted on the CPU); containers, per-read selection and scores
must equal the oracle's, and the device must decode them back.  The workload generator draws from every row alone.

The last tests run idn_gpu_decompress_reads, the dense-index form of the decoder, on the compat containers above and
on malformed indexes.
"""
from concurrent.futures import ThreadPoolExecutor
import os

import numpy as np
import pytest

from gpu_util import blocks_of, parse_compat_block, parse_spec, synth_on_device, upload

COMPAT, NATIVE = 1, 2
BLOCK = 4 * 1024 * 1024
TOTAL = 1 << 14
THREADS = os.cpu_count() or 8


# ---- adversarial rows ------------------------------------------------------------------------------------------------
def _from_starts(starts):
    s = np.asarray(starts, dtype=np.int64)
    f = np.diff(np.append(s, TOTAL))
    assert s[0] == 0 and (f >= 1).all(), "starts must begin at 0 and increase"
    return f


def _pinned(nsym, pins):
    """starts of nsym symbols with start(s) = pins[s]; the others spread evenly between their pinned neighbours"""
    pins = dict(pins)
    pins.setdefault(0, 0)
    pins[nsym] = TOTAL
    keys = sorted(pins)
    starts = np.zeros(nsym, dtype=np.int64)
    for a, b in zip(keys, keys[1:]):
        starts[a:b] = np.linspace(pins[a], pins[b], b - a, endpoint=False).astype(np.int64)
    return _from_starts(starts)


def _fill(rng, nsym, values):
    """nsym - 1 frequencies drawn from `values` while they fit, then 1s; the last symbol takes the rest"""
    f = []
    for _ in range(nsym - 1):
        v = int(rng.choice(values))
        f.append(v if sum(f) + v + (nsym - 1 - len(f)) <= TOTAL - 1 else 1)
    return np.asarray(f + [TOTAL - sum(f)])


def q_rows():
    rows = {}
    for p in (0, 47, 93):
        f = np.ones(94, dtype=np.int64)
        f[p] = TOTAL - 93
        rows[f"dominant{p}"] = f
    rows["uniform_174_175"] = np.asarray([175] * 28 + [174] * 66)
    rows["uniform_174_175_rev"] = rows["uniform_174_175"][::-1].copy()
    units = np.asarray([2] * 34 + [1] * 60)  # 128 units of 128 slots: every start on a multiple of 128
    edges = np.concatenate([[0], np.cumsum(units)[:-1]]) * 128
    rows["starts_128k"] = _from_starts(edges)
    rows["starts_128k_minus1"] = _from_starts(np.where(edges > 0, edges - 1, 0))
    rows["starts_128k_plus1"] = _from_starts(np.where(edges > 0, edges + 1, 0))
    for n in range(3, 9):
        # four clusters: the owner s0 of slot 128 k (s0 = 0 .. 3 mod 4, starting on or 3 slots before the bucket) and n
        # starts inside bucket k, the next start in bucket k + 1
        pins = {}
        for c in range(4):
            s0, k = 20 * c + 8 + c, 25 + 25 * c
            pins[s0] = 128 * k - (3 if c % 2 else 0)
            for t in range(1, n + 1):
                pins[s0 + t] = 128 * k + 13 * t
            pins[s0 + n + 1] = 128 * (k + 1) + 50
        rows[f"bucket_{n}_starts"] = _pinned(94, pins)
    rng = np.random.default_rng(1234)
    rows["pow2"] = _fill(rng, 94, [1 << k for k in range(13)])
    rows["pow2_pm1"] = _fill(rng, 94, [(1 << k) + d for k in range(1, 12) for d in (-1, 1)])
    f = np.ones(94, dtype=np.int64)
    f[20] = f[70] = (TOTAL - 92) // 2
    rows["two_dominant"] = f
    p = rng.dirichlet(np.full(94, 0.02))
    f = np.maximum(1, np.floor(p * TOTAL)).astype(np.int64)
    f[np.argmax(f)] += TOTAL - f.sum()
    rows["dirichlet_0.02"] = f
    return rows


def acid_rows():
    rows = {}
    for s in range(5):
        f = np.ones(5, dtype=np.int64)
        f[s] = TOTAL - 4
        rows[f"dominant{s}"] = f
    rows["adjacent_middle"] = np.asarray([8190, 1, 1, 1, 8191])
    rows["adjacent_low"] = np.asarray([1, 1, 1, 8190, 8191])
    rows["adjacent_pairs"] = np.asarray([5000, 1, 6000, 1, 5382])
    rows["pow2_desc"] = np.asarray([8192, 4096, 2048, 1024, 1024])
    rows["pow2_asc"] = np.asarray([1024, 1024, 2048, 4096, 8192])
    rows["pow2_flat"] = np.asarray([4096, 4096, 4096, 2048, 2048])
    rows["pow2_pm1"] = np.asarray([4095, 4097, 2047, 2049, 4096])
    rows["uniform"] = np.asarray([3277, 3277, 3277, 3277, 3276])
    return rows


Q_ROWS, A_ROWS = q_rows(), acid_rows()


def probs_of(rows):
    return np.stack([np.asarray(f, dtype=np.float32) / np.float32(TOTAL) for f in rows.values()])


def starts_of(f):
    return np.concatenate([[0], np.cumsum(f)[:-1]]).astype(np.int64)


def test_rows_are_exact_under_the_quantiser(O):
    """probs = f / 16384 in f32 gives back f from the pinned quantiser (and from the oracle's model tables)"""
    for rows in (Q_ROWS, A_ROWS):
        for name, f in rows.items():
            assert len(f) in (5, 94) and f.min() >= 1 and f.sum() == TOTAL, name
            p = (np.asarray(f, dtype=np.float32) / np.float32(TOTAL)).astype(np.float32)
            assert np.array_equal(O.quantise(p).astype(np.int64), starts_of(f)), name
        mtype = O.ACID if rows is A_ROWS else O.QSCORE
        md = O.ModelData.from_contexts(mtype, "generic_ao0_qo1_pb0", [([k], p) for k, p in enumerate(probs_of(rows))])
        tab = O.Model(md).cum_table().astype(np.int64)
        for r, f in enumerate(rows.values()):
            assert np.array_equal(tab[r + 1, :-1], starts_of(f)) and tab[r + 1, -1] == TOTAL


# ---- the row layouts of idn_device.cuh, restated, over all 16 384 slots -------------------------------------------------
def q_layout(f):
    """compact row: lut[k] = (symbol owning slot 128 k) >> 2, window g = starts of 4g .. 4g+7 (2^14 from symbol 94 on);
    window row entry k = {s0 = symbol owning slot 128 k, starts of s0 .. s0+6}"""
    st = np.append(starts_of(f), [TOTAL] * 16)
    owner = np.searchsorted(st[:94], 128 * np.arange(128), side="right") - 1
    lut = owner >> 2
    wins = np.stack([st[4 * g:4 * g + 8] for g in range(24)])
    winrows = np.stack([np.concatenate([[s0], st[s0:s0 + 7]]) for s0 in owner])
    return lut, wins, winrows


def q_search(f):
    """-> (symbol of every slot, window advances of q_find, j of q_find_win, whether q_find_win falls back)"""
    lut, wins, winrows = q_layout(f)
    slot = np.arange(TOTAL)
    g = lut[slot >> 7].astype(np.int64)
    adv = np.zeros(TOTAL, dtype=np.int64)
    while True:
        more = wins[g, 7] <= slot  # the last start of the window is still <= slot: next window
        if not more.any():
            break
        g = g + more
        adv += more
    j = (wins[g] <= slot[:, None]).sum(axis=1) - 1
    sym = 4 * g + j
    e = winrows[slot >> 7]
    jw = (e[:, 2:8] <= slot[:, None]).sum(axis=1)
    fallback = jw == 6
    truth = np.searchsorted(starts_of(f), slot, side="right") - 1
    assert np.array_equal(sym, truth), "restated q_find disagrees with the frequencies"
    assert np.array_equal((e[:, 0] + jw)[~fallback], truth[~fallback]), "restated q_find_win disagrees"
    return truth, adv, jw, fallback


def test_rows_reach_every_table_branch():
    advances, jws, fallbacks, edge = set(), set(), set(), set()
    for f in Q_ROWS.values():
        _, adv, jw, fb = q_search(f)
        advances |= set(np.unique(adv).tolist())
        jws |= set(np.unique(jw).tolist())
        fallbacks |= set(np.unique(fb).tolist())
        edge |= set((starts_of(f)[1:] % 128).tolist()) & {0, 1, 127}
    assert advances == set(range(23)), f"q_find advances reached: {sorted(advances)}"
    assert jws == set(range(7)) and fallbacks == {False, True}, (sorted(jws), fallbacks)
    assert edge == {0, 1, 127}, "starts on a bucket edge and one slot to either side"
    # acid_find: symbol = number of cum[1..4] <= slot; every outcome, and every symbol somewhere with frequency 1 (its
    # one slot is the boundary itself)
    outcomes, freq1 = set(), set()
    for f in A_ROWS.values():
        c = starts_of(f)[1:]
        slot = np.arange(TOTAL)
        sym = (c[None, :] <= slot[:, None]).sum(axis=1)
        assert np.array_equal(sym, np.searchsorted(starts_of(f), slot, side="right") - 1)
        outcomes |= set(np.unique(sym).tolist())
        freq1 |= set(np.flatnonzero(f == 1).tolist())
    assert outcomes == freq1 == set(range(5))


# ---- context specs of a read, vectorised (checked against the oracle's generator) ----------------------------------------
def spec_stream(name, read_off, acids, quals):
    """ContextSpecGenerator::current_context at every position of every read (context_spec.rs:377-389, 508-529)"""
    kind, ao, qo, pb, qmax = parse_spec(name)
    a, q = acids.astype(np.int64), quals.astype(np.int64)
    if kind == 1:
        ba, bq = 4, qmax
        z = (a == 0) | (q == 0)
        va, vq = np.where(z, 0, a - 1), np.where(z, 0, q * qmax // 94)
    else:
        ba, bq, va, vq = 5, 94, a, q
    lens = np.diff(read_off.astype(np.int64))
    i = np.arange(len(a)) - np.repeat(read_off[:-1].astype(np.int64), lens)
    L = np.repeat(lens, lens)

    def state(v, base, order):
        s = np.zeros(len(v), dtype=np.int64)
        for k in range(order):  # digit k = the symbol k + 1 positions back, 0 before the read starts
            sh = np.concatenate([np.zeros(k + 1, dtype=np.int64), v[:len(v) - k - 1]])[:len(v)]
            s += np.where(i > k, sh, 0) * base ** k
        return s
    abits = (ba ** ao - 1).bit_length()  # IntQueue::num_bits
    sa, sq = state(va, ba, ao), state(vq, bq, qo)
    pos = (i << pb) // np.maximum(L, 1)
    return ((((sq << abits) | sa) << pb) | pos).astype(np.int64)


def rand_reads(O, seed, total, long_reads=6):
    """uniformly random symbols; lengths 0 .. 300 plus a few reads of about 5 000 symbols"""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 301, size=int(total // 150))
    lens = np.insert(lens, rng.integers(0, len(lens), size=long_reads), rng.integers(4900, 5100, size=long_reads))
    ro = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=ro[1:])
    S = int(ro[-1])
    return O.Reads(ro, rng.integers(0, 5, size=S).astype(np.uint8), rng.integers(0, 94, size=S).astype(np.uint8), None, None)


def map_specs(specs, n_ctx, salt):
    """multiplicative hash of the spec (its low bits are the position bin): about 1 in 8 unmapped (-1), the rest onto
    0 .. n_ctx - 1"""
    h = (specs.astype(np.uint64) + np.uint64(salt)) * np.uint64(0x9E3779B97F4A7C15)
    u = (h >> np.uint64(40)).astype(np.int64)  # 24 bits
    return np.where(u < (1 << 21), -1, (u - (1 << 21)) * n_ctx // (7 << 21))


# (acid spec type, q-score spec type, expected kernel variant)
CONFIGS = {
    "SP0": ("light_ao8_qo0_pb0_qm1", "generic_ao0_qo2_pb6", 0),
    "SP1": ("light_ao8_qo0_pb0_qm1", "generic_ao2_qo1_pb6", 1),
    "SP2": ("generic_ao8_qo0_pb0", "light_ao0_qo4_pb0_qm16", 2),
    "SP3": ("light_ao4_qo3_pb2_qm8", "light_ao0_qo4_pb3_qm16", 3),
    "SP4": ("generic_ao4_qo1_pb2", "light_ao0_qo4_pb3_qm16", 4),
    "SP5": ("generic_ao8_qo0_pb0", "light_ao2_qo4_pb2_qm8", 5),
    "SP6": ("generic_ao8_qo0_pb0", "light_ao0_qo3_pb0_qm32", 6),
    "SP7": ("generic_ao8_qo0_pb0", "light_ao0_qo4_pb3_qm16", 7),
    "dyn_pb": ("generic_ao4_qo0_pb6", "light_ao2_qo3_pb2_qm16", -1),  # DynSpecs, position bits on both sides
    "big_dense_acid": ("light_ao8_qo1_pb2_qm16", "generic_ao0_qo3_pb0", -1),  # 2^22 acid specs: no adirect / aenc
    "hashed": ("generic_ao8_qo0_pb4", "generic_ao3_qo3_pb0", -1),  # 2^23 and 2^27 specs: hashed maps
}
DENSE_LIMIT = 1 << 22


def make_model(O, mtype, name, rows, reads, salt, reached):
    """contexts = the adversarial rows in a salted order; dense spec spaces list every spec, hashed ones the specs the
    reads reach (a random half of them mapped).  reached: spec type -> the sorted specs the reads reach (cache)"""
    probs = probs_of(rows)
    n = len(probs)
    probs = probs[np.random.default_rng(salt).permutation(n)]
    if O.spec_num(name) <= DENSE_LIMIT:
        specs = np.arange(O.spec_num(name), dtype=np.int64)
        ctx = map_specs(specs, n, salt)
    else:
        if name not in reached:
            reached[name] = np.unique(spec_stream(name, reads.read_off, reads.acids, reads.quals))
        specs = np.sort(np.random.default_rng(salt).choice(reached[name], size=len(reached[name]) // 2, replace=False))
        ctx = map_specs(specs, n, salt) % n
    keys, ctx = specs[ctx >= 0].astype(np.uint32), ctx[ctx >= 0].astype(np.uint32)
    return O.Model(O.ModelData(mtype, name, probs, keys, ctx, O.make_identifier(mtype, name, probs, keys, ctx)))


def rows_of(model, specs):
    """context row (0 = dummy) of every spec under `model`"""
    keys, ctx = model.md.spec_keys.astype(np.int64), model.md.spec_ctx.astype(np.int64)
    i = np.minimum(np.searchsorted(keys, specs), len(keys) - 1)
    return np.where(keys[i] == specs, ctx[i] + 1, 0)


@pytest.fixture(scope="module")
def cfg_data(O):
    """config -> (reads, [acid model, q-score model], [second acid model, second q-score model]); built on first use"""
    cache = {}

    def get(name):
        if name not in cache:
            an, qn, _ = CONFIGS[name]
            reads = rand_reads(O, 100 + list(CONFIGS).index(name), 1.5 * BLOCK)
            reached = {}
            pair = [make_model(O, O.ACID, an, A_ROWS, reads, 11, reached), make_model(O, O.QSCORE, qn, Q_ROWS, reads, 12, reached)]
            alt = [make_model(O, O.ACID, an, A_ROWS, reads, 21, reached), make_model(O, O.QSCORE, qn, Q_ROWS, reads, 22, reached)]
            cache[name] = (reads, pair, alt)
        return cache[name]
    return get


def test_spec_restatement_matches_the_oracle(O):
    rng = np.random.default_rng(3)
    lens = np.concatenate([[0, 1, 2, 9], rng.integers(1, 200, size=40)])
    ro = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=ro[1:])
    S = int(ro[-1])
    a, q = rng.integers(0, 5, size=S).astype(np.uint8), rng.integers(0, 94, size=S).astype(np.uint8)
    for name in sorted({n for an, qn, _ in CONFIGS.values() for n in (an, qn)}):
        got = spec_stream(name, ro, a, q)
        want = []
        for r in range(len(lens)):
            g = O.Generator(name, int(lens[r]))
            for i in range(int(ro[r]), int(ro[r + 1])):
                want.append(g.current_context())
                g.update(int(a[i]), int(q[i]))
        assert np.array_equal(got, np.asarray(want, dtype=np.int64)), name
        assert got.max() < O.spec_num(name)


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_reads_code_every_row_symbol_pair(O, cfg_data, cfg):
    """Over the first ~1 M symbols every (row, symbol) pair of every adversarial row is coded at least 5 times, in
    both models of the pair (the second pair's rows are the same, in another order)."""
    an, qn, _ = CONFIGS[cfg]
    reads, pair, alt = cfg_data(cfg)
    r_end = int(np.searchsorted(reads.read_off, 1 << 20))
    ro = reads.read_off[:r_end + 1]
    S = int(ro[-1])
    for name, m, sym, nsym in ((an, pair[0], reads.acids, 5), (qn, pair[1], reads.quals, 94),
                               (an, alt[0], reads.acids, 5), (qn, alt[1], reads.quals, 94)):
        rows = rows_of(m, spec_stream(name, ro, reads.acids[:S], reads.quals[:S]))
        cnt = np.bincount(rows * nsym + sym[:S].astype(np.int64), minlength=(m.md.n_ctx + 1) * nsym).reshape(-1, nsym)
        assert cnt[0].sum() > 0.05 * S, "the dummy row is used as well"
        low = np.argwhere(cnt[1:] < 5)
        assert not len(low), f"{name}: row {low[0][0] + 1} symbol {low[0][1]} coded {cnt[1:][tuple(low[0])]} times"


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gctx():
    from idencomp_b200 import capi
    ctx = capi.Context(0)
    ctx.set_pipeline_blocks(1 << 16)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def cfg_dev(gctx, O, cfg_data):
    """config -> dict(reads, models, handles (acid, q, acid', q'), bf, compat=(out, block_off, crc) once computed)"""
    cache = {}

    def get(name):
        if name not in cache:
            reads, pair, alt = cfg_data(name)
            models = pair + alt
            cache[name] = dict(reads=reads, models=models, handles=[upload(gctx, O, m) for m in models],
                               bf=blocks_of(reads, BLOCK))
        return cache[name]
    yield get
    for d in cache.values():
        for h in d["handles"]:
            gctx.release_model(h)


def compat_file(models, out):
    return b"IDENCOMP\x01" + bytes([1, 0, len(models)]) + b"".join(m.md.identifier for m in models) + out.tobytes() + b"\x00" * 8


def decode(gctx, out, block_off, crc, handles, mode, reads):
    doff = np.append(block_off[:-1] + 8, block_off[-1]).astype(np.uint64)
    dlen = (block_off[1:] - block_off[:-1] - 8).astype(np.uint32)
    ro, a, q = gctx.decompress_blocks(out, doff, crc, handles, block_len=dlen, mode=mode, reads_cap=reads.n_reads,
                                      symbols_cap=int(reads.read_off[-1]))
    assert np.array_equal(ro, reads.read_off), "decoded read lengths differ"
    assert np.array_equal(a, reads.acids) and np.array_equal(q, reads.quals), "decoded symbols differ"


def compat_of(gctx, d):
    """the device's compat container of the adversarial pair alone (cached for the per-read decoder tests)"""
    if "compat" not in d:
        r = d["reads"]
        out, block_off, crc, _ = gctx.compress_blocks(r.read_off, r.acids, r.quals, d["bf"], d["handles"][:2])
        d["compat"] = (out, block_off, crc)
    return d["compat"]


def check_native(O, gctx, d, models, handles, lane_syms):
    reads, bf = d["reads"], d["bf"]
    gctx.set_lane_symbols(lane_syms)
    try:
        out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, handles, mode=NATIVE)
    finally:
        gctx.set_lane_symbols(2048)
    with ThreadPoolExecutor(THREADS) as ex:
        expect = list(ex.map(lambda b: O.compress_native_block(models, reads, int(bf[b]), int(bf[b + 1] - bf[b]), lane_syms=lane_syms,
                                                               include_identifiers=False), range(len(bf) - 1)))
    for b, (data, ecrc) in enumerate(expect):
        blk = out[int(block_off[b]):int(block_off[b + 1])].tobytes()
        assert int.from_bytes(blk[0:4], "big") == len(data) and blk[8:] == data, f"native block {b} differs"
        assert int.from_bytes(blk[4:8], "big") == ecrc == int(crc[b]), f"native block {b} crc"
    decode(gctx, out, block_off, crc, handles, NATIVE, reads)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_compat_vs_oracle(gctx, O, cfg_dev, cfg):
    """the whole .idn == the oracle's, and back; the pair launches the kernel variant it is meant to cover"""
    d = cfg_dev(cfg)
    assert gctx.kernel_variant(*d["handles"][:2]) == CONFIGS[cfg][2]
    assert len(d["bf"]) - 1 == 2
    out, block_off, crc = compat_of(gctx, d)
    ref = O.compress(d["models"][:2], d["reads"], include_identifiers=False, threads=THREADS)
    assert compat_file(d["models"][:2], out) == ref, "device container differs from the oracle's"
    decode(gctx, out, block_off, crc, d["handles"][:2], COMPAT, d["reads"])


@pytest.mark.gpu
@pytest.mark.parametrize("lane_syms", [256, 2048])
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_native_vs_oracle(gctx, O, cfg_dev, cfg, lane_syms):
    d = cfg_dev(cfg)
    check_native(O, gctx, d, d["models"][:2], d["handles"][:2], lane_syms)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [COMPAT, NATIVE], ids=["compat", "native"])
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_selection_vs_oracle(gctx, O, cfg_dev, cfg, mode):
    """per-read (compat) / per-lane (native, quantum 256) choice between the adversarial pair and a second pair of the
    same spec types with the rows in another order: the list kernels run on these rows"""
    d = cfg_dev(cfg)
    reads = d["reads"]
    order = [0, 2, 1, 3]  # acid models first
    models, handles = [d["models"][k] for k in order], [d["handles"][k] for k in order]
    if mode == COMPAT:
        out, block_off, crc, st = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, d["bf"], handles)
        assert compat_file(models, out) == O.compress(models, reads, include_identifiers=False, threads=THREADS)
        assert st["acid_switches"] > 100 and st["q_switches"] > 100, "both pairs are chosen"
        decode(gctx, out, block_off, crc, handles, COMPAT, reads)
    else:
        check_native(O, gctx, d, models, handles, 256)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_scores_vs_oracle(gctx, O, cfg_dev, cfg):
    d = cfg_dev(cfg)
    reads = d["reads"]
    sizes = gctx.score((reads.read_off, reads.acids, reads.quals), d["handles"])
    rows = np.random.default_rng(8).choice(reads.n_reads, size=300, replace=False)
    rows = np.append(rows, np.flatnonzero(np.diff(reads.read_off.astype(np.int64)) > 4000))
    for r in rows:
        s0, s1 = int(reads.read_off[r]), int(reads.read_off[r + 1])
        for k, m in enumerate(d["models"]):
            assert int(sizes[r, k]) == O.score_read(m, reads.acids[s0:s1], reads.quals[s0:s1]), (cfg, int(r), k)


@pytest.mark.gpu
def test_sampler_draws_every_slot_of_every_row(gctx, O):
    """idn_gpu_synth_reads_dev resolves uniform slots through q_find (compact row) and acid_find: with one dummy-spec
    model per row, 300 000 draws per row equal the oracle's sampler and hit every symbol (a given slot goes
    unsampled with probability e^-18)"""
    qn, an = list(Q_ROWS), list(A_ROWS)
    ro = np.arange(0, 300_001, 1000, dtype=np.uint64)
    for i in range(max(len(qn), len(an))):
        fa, fq = A_ROWS[an[i % len(an)]], Q_ROWS[qn[i % len(qn)]]
        am = O.Model(O.ModelData.from_contexts(O.ACID, "dummy", [([0], probs_of({0: fa})[0])]))
        qm = O.Model(O.ModelData.from_contexts(O.QSCORE, "dummy", [([0], probs_of({0: fq})[0])]))
        ha, hq = upload(gctx, O, am), upload(gctx, O, qm)
        try:
            a, q = synth_on_device(gctx, ha, hq, ro, seed=500 + i, n_ppm=0)
        finally:
            gctx.release_model(ha)
            gctx.release_model(hq)
        want = O.synth_reads(am, qm, ro, 0, 500 + i, 0, threads=THREADS)
        assert np.array_equal(a, want.acids) and np.array_equal(q, want.quals), (an[i % len(an)], qn[i % len(qn)])
        assert (np.bincount(a, minlength=5) > 0).all() and (np.bincount(q, minlength=94) > 0).all()


# ---- idn_gpu_decompress_reads ------------------------------------------------------------------------------------------
READS_CFGS = ["SP0", "SP1", "SP3", "dyn_pb", "big_dense_acid", "hashed"]


@pytest.fixture(scope="module")
def read_index(gctx, cfg_dev):
    """The compat containers of several configs back to back in one payload, and the per-read index a CPU walk of their
    slices gives: (payload, index columns, models list, expected acids / quals per read)"""
    payload, cols, models, exp = [], {k: [] for k in ("pay_off", "pay_len", "seq_len", "am", "qm")}, [], []
    base = 0
    for cfg in READS_CFGS:
        d = cfg_dev(cfg)
        out, block_off, _ = compat_of(gctx, d)
        m0 = len(models)
        models += d["handles"][:2]
        r = 0
        for b in range(len(block_off) - 1):
            data = out[int(block_off[b]) + 8:int(block_off[b + 1])].tobytes()
            ga, gq, _, _, po, pl, sl = parse_compat_block(data, [True, False], offsets=True)
            assert (ga == 0).all() and (gq == 1).all()
            cols["pay_off"].append(po + np.uint64(base + int(block_off[b]) + 8))
            cols["pay_len"].append(pl)
            cols["seq_len"].append(sl)
            cols["am"].append(ga + m0)
            cols["qm"].append(gq + m0)
            r += len(sl)
        reads = d["reads"]
        assert r == reads.n_reads
        exp += [(reads.acids[int(reads.read_off[i]):int(reads.read_off[i + 1])],
                 reads.quals[int(reads.read_off[i]):int(reads.read_off[i + 1])]) for i in range(reads.n_reads)]
        payload.append(out)
        base += len(out)
    cols = {k: np.concatenate(v) for k, v in cols.items()}
    return np.concatenate(payload), cols, models, exp


def _take(cols, perm):
    return {k: v[perm] for k, v in cols.items()}


def _call(gctx, payload, c, models, **kw):
    return gctx.decompress_reads(payload, c["pay_off"], c["pay_len"], c["seq_len"], c["am"], c["qm"], models, **kw)


@pytest.mark.gpu
def test_decompress_reads_shuffled(gctx, read_index):
    """every read of six configs' compat containers, in a shuffled order, through one call"""
    payload, cols, models, exp = read_index
    perm = np.random.default_rng(4).permutation(len(exp))
    c = _take(cols, perm)
    assert np.array_equal(c["seq_len"], [len(exp[i][0]) for i in perm])
    oo, a, q, st = _call(gctx, payload, c, models)
    assert (st == 0).all(), f"read_status of read {perm[np.flatnonzero(st)[0]]}: {st[st != 0][0]}"
    assert np.array_equal(a, np.concatenate([exp[i][0] for i in perm]))
    assert np.array_equal(q, np.concatenate([exp[i][1] for i in perm]))


@pytest.mark.gpu
def test_decompress_reads_reports_bad_payloads(gctx, read_index):
    """one payload a byte short and another a byte long: SerializeError, and read_status flags exactly those two"""
    from idencomp_b200.capi import IdnGpuError
    payload, cols, models, _ = read_index
    rng = np.random.default_rng(6)
    perm = rng.permutation(len(cols["seq_len"]))[:5000]
    c = _take(cols, perm)
    live = np.flatnonzero((c["seq_len"] > 20) & (c["pay_off"] + c["pay_len"] + 1 < len(payload)))
    short, long_ = int(live[10]), int(live[20])
    c["pay_len"][short] -= 1
    c["pay_len"][long_] += 1
    with pytest.raises(IdnGpuError) as e:
        _call(gctx, payload, c, models)
    assert e.value.kind == "SerializeError"
    assert np.flatnonzero(e.value.read_status).tolist() == sorted([short, long_])


@pytest.mark.gpu
def test_decompress_reads_argument_errors(gctx, read_index):
    from idencomp_b200.capi import IdnGpuError
    payload, cols, models, _ = read_index
    c0 = _take(cols, np.arange(200))

    def refused(kind, out_off=None, **kw):
        c = {k: v.copy() for k, v in c0.items()}
        for k, (i, v) in kw.items():
            c[k][i] = v
        with pytest.raises(IdnGpuError) as e:
            _call(gctx, payload, c, models, out_off=out_off)
        assert e.value.kind == kind, (kw, e.value)

    scan = np.zeros(201, dtype=np.uint64)
    np.cumsum(c0["seq_len"], out=scan[1:])
    for r in (0, 7, 200):
        bad = scan.copy()
        bad[r] += 1
        refused("InvalidArgument", out_off=bad)
    refused("InvalidModelIndex", am=(3, len(models)))
    refused("InvalidModelIndex", qm=(5, 255))
    refused("InvalidModelIndex", am=(9, 1))  # a q-score model in the acid column
    refused("InvalidModelIndex", qm=(9, 0))
    refused("SerializeError", pay_off=(11, len(payload) - int(c0["pay_len"][11]) + 1))
    refused("SerializeError", pay_off=(12, (1 << 64) - 4), pay_len=(12, 8))  # pay_off + pay_len wraps past 2^64
    oo, a, q, st = gctx.decompress_reads(payload, np.zeros(0), np.zeros(0), np.zeros(0), np.zeros(0), np.zeros(0), models)
    assert len(a) == len(q) == len(st) == 0 and oo.tolist() == [0]

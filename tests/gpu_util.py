"""Helpers shared by the parity tests: feed oracle-side model data through the C-ABI; synthetic models per spec type;
the bundled same-sequencer model pairs and model-driven reads drawn on the device."""
import ctypes as C
import re

import numpy as np


def parse_spec(name: str):
    """spec type name -> (kind, ao, qo, pb, qmax)   (idencomp-macros/src/lib.rs:166-196)"""
    if name == "dummy":
        return 0, 0, 0, 0, 0
    m = re.fullmatch(r"generic_ao(\d+)_qo(\d+)_pb(\d+)", name)
    if m:
        return (0, *map(int, m.groups()), 0)
    m = re.fullmatch(r"light_ao(\d+)_qo(\d+)_pb(\d+)_qm(\d+)", name)
    if m:
        return (1, *map(int, m.groups()))
    raise ValueError(name)


def upload(gctx, O, model) -> int:
    """Upload an oracle Model (its integer tables come from the pinned quantiser) through idn_gpu_model_upload."""
    md = model.md
    kind, ao, qo, pb, qmax = parse_spec(md.spec_name)
    return gctx.upload_model(md.mtype, kind, ao, qo, pb, qmax, model.cum_table(), md.spec_keys, md.spec_ctx)


def blocks_of(reads, max_block_total_len):
    """IdnCompressor::add_sequence block forming (idn/compressor.rs:517-540): block_first_read."""
    first = [0]
    cur = 0
    for r in range(reads.n_reads):
        ln = int(reads.read_off[r + 1] - reads.read_off[r])
        if cur + ln > max_block_total_len and cur > 0:
            first.append(r)
            cur = 0
        cur += ln
    first.append(reads.n_reads)
    return np.asarray(first, dtype=np.uint32)


# ---- every legal context-spec type (the model!{} list, context_spec.rs:532-599): dummy + 23 generic + 26 light ----
GENERIC = [(1, 0, 0), (2, 0, 0), (4, 0, 0), (8, 0, 0), (0, 1, 0), (0, 2, 0), (0, 3, 0), (0, 0, 2), (0, 0, 4), (0, 0, 8), (4, 1, 2),
           (1, 3, 2), (2, 1, 6), (6, 2, 0), (3, 3, 0), (8, 0, 4), (4, 0, 3), (4, 0, 6), (0, 2, 6), (0, 3, 3), (4, 2, 6), (5, 2, 4),
           (3, 3, 4)]
LIGHT = [(4, 1, 2, 16), (8, 1, 2, 16), (8, 0, 0, 1), (0, 3, 3, 8), (0, 3, 3, 16), (0, 4, 3, 8), (0, 4, 3, 16), (0, 4, 0, 8),
         (0, 4, 0, 16), (3, 3, 0, 8), (3, 3, 0, 16), (2, 3, 2, 8), (0, 4, 2, 8), (2, 3, 2, 16), (0, 4, 2, 16), (2, 4, 2, 8),
         (4, 3, 4, 16), (4, 3, 2, 8), (0, 3, 0, 4), (0, 3, 0, 8), (0, 3, 0, 16), (0, 3, 0, 32), (4, 4, 4, 8), (4, 4, 4, 16),
         (5, 4, 4, 16), (3, 5, 4, 16)]
SPEC_NAMES = (["dummy"] + [f"generic_ao{a}_qo{q}_pb{p}" for a, q, p in GENERIC] +
              [f"light_ao{a}_qo{q}_pb{p}_qm{m}" for a, q, p, m in LIGHT])
assert len(SPEC_NAMES) == 50


def toy_reads(O, seed, n=48):
    """short ragged reads with few distinct quality values and some N / q = 0, so that contexts repeat"""
    rng = np.random.default_rng(seed)
    seqs = [("", [], [])]
    for _ in range(n):
        ln = int(rng.integers(1, 120))
        a = rng.choice([0, 1, 2, 3, 4], size=ln, p=[0.04, 0.3, 0.22, 0.22, 0.22])
        q = rng.choice([0, 2, 11, 25, 37, 40, 93], size=ln, p=[0.03, 0.07, 0.2, 0.3, 0.25, 0.1, 0.05])
        seqs.append(("", a, q))
    return O.Reads.from_lists(seqs)


def synthetic_model(O, mtype, spec_name, reads, seed, n_ctx=3):
    """a model of `spec_name` whose contexts own the most frequent specs of `reads` (several specs per context, i.e. binned),
    with skewed probabilities incl. exact zeros (the zero-frequency fix-up of the quantiser)"""
    rng = np.random.default_rng(seed)
    counts = {}
    for r in range(reads.n_reads):
        s0, s1 = int(reads.read_off[r]), int(reads.read_off[r + 1])
        g = O.Generator(spec_name, s1 - s0)
        for i in range(s0, s1):
            sp = g.current_context()
            counts[sp] = counts.get(sp, 0) + 1
            g.update(int(reads.acids[i]), int(reads.quals[i]))
    top = [sp for sp, _ in sorted(counts.items(), key=lambda kv: (-kv[1], kv[0]))[:3 * n_ctx]]
    nsym = 5 if mtype == O.ACID else 94
    ctxs = []
    for k in range(min(n_ctx, len(top))):
        p = rng.dirichlet(np.full(nsym, 0.3)).astype(np.float32)
        p[rng.integers(0, nsym)] = 0.0
        ctxs.append((sorted(top[k::n_ctx]), (p / p.sum()).tolist()))
    return O.Model(O.ModelData.from_contexts(mtype, spec_name, ctxs))


# (acid model, q-score model, read lengths, expected kernel variant): the same-sequencer pairs of models/ (models.md)
PAIRS = {
    "hiseq2000": ("ERR174310__human__illumina_hiseq_2000__acids", "SRR2962693__human__illumina_hiseq_2500__q_scores", (100, 100), 0),
    "hiseq2500_human": ("SRR2962693__human__illumina_hiseq_2500__acids", "SRR2962693__human__illumina_hiseq_2500__q_scores", (70, 101), 0),
    "hiseq2500_b_stabilis": ("SRR19549058__b_stabilis__illumina_hiseq_2500__acids", "SRR19549058__b_stabilis__illumina_hiseq_2500__q_scores", (125, 125), 0),
    "novaseq_human": ("SRR8861483__human__illumina_novaseq_6000__acids", "SRR8861483__human__illumina_novaseq_6000__q_scores", (150, 150), 1),
    "sequel2": ("m64187e__sars_cov_2__sequel_ii_e__acids", "m64187e__sars_cov_2__sequel_ii_e__q_scores", (10_000, 20_000), 2),
    "novaseq_cat": ("SRR18908372__cat__illumina_novaseq_6000__acids", "SRR18908372__cat__illumina_novaseq_6000__q_scores", (151, 151), 3),
    "hiseq2500_cat": ("SRR5373739__cat__illumina_hiseq_2500__acids", "SRR5373739__cat__illumina_hiseq_2500__q_scores", (90, 126), 4),
    "iseq100": ("ERR5462922__ebov__illumina_iseq_100__acids", "ERR5462922__ebov__illumina_iseq_100__q_scores", (151, 151), 5),
    "hiseq2500_e_coli": ("SRR16141966__e_coli__illumina_hiseq_2500__acids", "SRR16141966__e_coli__illumina_hiseq_2500__q_scores", (100, 100), 6),
    "hiseq2500_pear": ("SRR19609907__pear__illumina_hiseq_2500__acids", "SRR19609907__pear__illumina_hiseq_2500__q_scores", (101, 101), 7),
    "hiseq2500_salmonella": ("SRR20210997__salmonella__illumina_hiseq_2500__acids", "SRR20210997__salmonella__illumina_hiseq_2500__q_scores", (100, 100), -1),
}


def parse_compat_block(data: bytes, is_acid, offsets=False):
    """Walk the slices of one compat block: 00 Identifiers (u32be len, u8 codec, data), 01 SwitchModel (u8 index),
    02 Sequence (u32be len, u32be seq_len, payload) (data.rs:46-84).  is_acid[i]: container model i is an acid model.
    -> (acid index, q-score index, acid switch before the read, q-score switch before the read), one entry per read;
    with offsets=True also (payload offset in `data`, payload length, sequence length) per read."""
    u32 = lambda pos: int.from_bytes(data[pos:pos + 4], "big")
    acid, qual, sw_a, sw_q, p_off, p_len, s_len = [], [], [], [], [], [], []
    cur_a = cur_q = -1
    pend_a = pend_q = False
    pos, n = 0, len(data)
    while pos < n:
        kind = data[pos]
        if kind == 0:
            pos += 6 + u32(pos + 1)
        elif kind == 1:
            idx = data[pos + 1]
            if is_acid[idx]:
                cur_a, pend_a = idx, True
            else:
                cur_q, pend_q = idx, True
            pos += 2
        elif kind == 2:
            acid.append(cur_a)
            qual.append(cur_q)
            sw_a.append(pend_a)
            sw_q.append(pend_q)
            pend_a = pend_q = False
            p_off.append(pos + 9)
            p_len.append(u32(pos + 1))
            s_len.append(u32(pos + 5))
            pos += 9 + u32(pos + 1)
        else:
            raise ValueError(f"unknown slice kind {kind} at byte {pos}")
    if pos != n:
        raise ValueError("the last slice overruns the block")
    out = (np.asarray(acid), np.asarray(qual), np.asarray(sw_a, dtype=bool), np.asarray(sw_q, dtype=bool))
    if offsets:
        out += (np.asarray(p_off, dtype=np.uint64), np.asarray(p_len, dtype=np.uint32), np.asarray(s_len, dtype=np.uint32))
    return out


def synth_on_device(gctx, ha, hq, read_off, seed, n_ppm=500):
    """Model-driven reads (idn_gpu_synth_reads_dev; equal to the oracle's sampler, test_gpu_parity.py) -> host arrays."""
    import torch
    S = int(read_off[-1])
    ro_d = torch.from_numpy(read_off.view(np.int64)).cuda()
    a_d = torch.zeros(S + 16, dtype=torch.uint8, device="cuda")
    q_d = torch.zeros(S + 16, dtype=torch.uint8, device="cuda")
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    gctx.check(gctx.L.idn_gpu_synth_reads_dev(gctx.h, ha, hq, ro_d.data_ptr(), len(read_off) - 1, 0, seed, n_ppm,
                                              a_d.data_ptr(), q_d.data_ptr(), sp))
    torch.cuda.synchronize()
    return a_d[:S].cpu().numpy(), q_d[:S].cpu().numpy()

"""Compat containers are assembled by kernels that only move or scan bytes: the block layout (a scan over the blocks)
and the slice copy from the encoder's scratch slots into the container (16-byte chunks, a group of lanes per read).
Their outputs are checked byte for byte against the oracle's containers and the serial layout rule.

Run on the B200 box: python -m pytest tests -m gpu
"""
import ctypes as C

import numpy as np
import pytest

from gpu_util import blocks_of, upload

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gctx():
    from idencomp_b200 import capi
    ctx = capi.Context(0)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def toy_handles(gctx, O, toy_models):
    return [upload(gctx, O, m) for m in toy_models]


def ragged_reads(O, seed, lengths):
    rng = np.random.default_rng(seed)
    return O.Reads.from_lists([("", rng.integers(0, 5, ln), rng.integers(0, 94, ln)) for ln in lengths])


def expected_blocks(O, models, reads, bf, fast):
    return [O.compress_block(models, reads, int(bf[b]), int(bf[b + 1] - bf[b]), include_identifiers=False, fast=fast)
            for b in range(len(bf) - 1)]


def check_blocks(out, block_off, crc, expect, prefix):
    """slices after the reserved prefix equal the oracle's block; block_off is the serial layout rule restated"""
    pos = 0
    for b, (data, ecrc, _) in enumerate(expect):
        assert int(block_off[b]) == pos, f"block {b} offset"
        blk = out[pos:pos + 8 + int(prefix[b]) + len(data)].tobytes()
        assert int.from_bytes(blk[0:4], "big") == int(prefix[b]) + len(data), f"block {b} length"
        assert int.from_bytes(blk[4:8], "big") == ecrc == int(crc[b]), f"block {b} crc"
        assert blk[8 + int(prefix[b]):] == data, f"block {b} slices differ"
        pos += 8 + int(prefix[b]) + len(data)
    assert int(block_off[len(expect)]) == pos


# ---- the slice copy ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("residue", range(16))
def test_copy_every_destination_residue(gctx, O, toy_models, toy_handles, residue):
    """The reserved prefix shifts every block body by `residue` bytes, and ragged reads (0 to 300 symbols) give every
    source residue: each read's slices land byte for byte where the oracle puts them, the block headers and the bytes
    between blocks untouched.  Non-fast mode puts SwitchModel slices in front of each block's first read."""
    lengths = np.random.default_rng(residue).integers(0, 300, 700)
    lengths[::37] = 0
    reads = ragged_reads(O, 100 + residue, lengths)
    bf = blocks_of(reads, 6000)
    prefix = np.full(len(bf) - 1, residue, dtype=np.uint32)
    prefix[::3] += 16
    expect = expected_blocks(O, toy_models, reads, bf, fast=False)
    out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, toy_handles, prefix_len=prefix)
    check_blocks(out, block_off, crc, expect, prefix)


def test_copy_switch_slices_empty_blocks_and_long_reads(gctx, O, model_data):
    """Per-read selection among 4 + 4 models (SwitchModel slices in the middle of blocks), empty blocks, zero-length reads,
    and reads of 3000-9000 symbols whose payloads are longer than a warp's 512 bytes of one pass."""
    from oracle import oracle as Om
    names = sorted(model_data)
    acids = [k for k in names if model_data[k].mtype == Om.ACID][:4]
    quals = [k for k in names if model_data[k].mtype == Om.QSCORE][:4]
    models = [O.Model(model_data[k]) for k in acids + quals]
    handles = [upload(gctx, O, m) for m in models]
    lengths = [100] * 300 + [0, 3000, 1, 9000, 0, 0, 150] + [100] * 200
    reads = ragged_reads(O, 5, lengths)
    bf = np.asarray([0, 0, 120, 120, 301, 307, 307, reads.n_reads], dtype=np.uint32)
    expect = expected_blocks(O, models, reads, bf, fast=False)
    out, block_off, crc, stats = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, handles)
    check_blocks(out, block_off, crc, expect, np.zeros(len(bf) - 1, dtype=np.uint32))
    assert stats["acid_switches"] + stats["q_switches"] > 7
    # fast mode: the 01 00 01 01 marker of every non-empty block, none in the empty ones
    expect = expected_blocks(O, models[:1] + models[4:5], reads, bf, fast=True)
    out, block_off, crc, _ = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, handles[:1] + handles[4:5], fast=True)
    check_blocks(out, block_off, crc, expect, np.zeros(len(bf) - 1, dtype=np.uint32))


def test_copy_respects_out_cap(gctx, O, toy_models, toy_handles):
    """At the required size the container is complete; one byte short the call reports NoSpace, no byte at or past
    out_cap is written, and the blocks before the last one are as in the complete container."""
    import torch
    from idencomp_b200 import capi
    reads = ragged_reads(O, 9, np.random.default_rng(9).integers(0, 200, 500))
    bf = blocks_of(reads, 8000)
    full, block_off, _, stats = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, toy_handles)
    need = stats["out_bytes"]
    assert need == len(full)
    with pytest.raises(capi.IdnGpuError) as ei:
        gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, toy_handles, out_cap=need - 1)
    assert ei.value.kind == "NoSpace"
    # the device entry point: the guard region past out_cap keeps its bytes
    dev = "cuda"
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ro = torch.from_numpy(reads.read_off.astype(np.int64)).to(dev)
    a_d = torch.from_numpy(np.append(reads.acids, np.zeros(16, np.uint8))).to(dev)
    q_d = torch.from_numpy(np.append(reads.quals, np.zeros(16, np.uint8))).to(dev)
    bf_d = torch.from_numpy(bf.astype(np.int32)).to(dev)
    b = capi.Batch()
    b.n_reads, b.n_symbols, b.n_blocks = reads.n_reads, int(reads.read_off[-1]), len(bf) - 1
    b.acids, b.quals, b.read_off, b.block_first_read = a_d.data_ptr(), q_d.data_ptr(), ro.data_ptr(), bf_d.data_ptr()
    hd = np.asarray(toy_handles, dtype=np.int32)
    for cap in (need, need - 1):
        out = torch.full((need + 64,), 0xA5, dtype=torch.uint8, device=dev)
        boff = torch.zeros(len(bf), dtype=torch.int64, device=dev)
        crc = torch.zeros(len(bf) - 1, dtype=torch.int32, device=dev)
        st = torch.zeros(8, dtype=torch.int64, device=dev)
        gctx.check(gctx.L.idn_gpu_compress_blocks_dev(gctx.h, C.byref(b), capi.MODE_COMPAT, hd.ctypes.data, 2, 0, None, out.data_ptr(),
                                                      cap, boff.data_ptr(), crc.data_ptr(), st.data_ptr(), sp))
        torch.cuda.synchronize()
        o = out.cpu().numpy()
        assert int(st[0]) == need
        assert (o[cap:] == 0xA5).all(), "bytes written at or past out_cap"
        if cap == need:
            assert o[:need].tobytes() == full.tobytes()
        else:  # every block but the last is complete
            lo = int(block_off[-2])
            assert o[:lo].tobytes() == full[:lo].tobytes()


# ---- the block layout ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_blocks", [0, 1, 1500])
@pytest.mark.parametrize("fast", [False, True])
def test_block_layout_against_the_serial_rule(gctx, O, toy_models, toy_handles, n_blocks, fast):
    """block_off[b + 1] = block_off[b] + 8 + prefix_len[b] + slices (+ 4 for the fast-mode marker of a non-empty block),
    with empty blocks among 1500 (more than one tile of the scan)."""
    from idencomp_b200.capi import IdnGpuError
    rng = np.random.default_rng(n_blocks)
    reads = ragged_reads(O, 7, rng.integers(0, 40, 2 * max(n_blocks, 1)))
    if n_blocks == 0:  # a batch without blocks is refused before any kernel runs
        with pytest.raises(IdnGpuError) as ei:
            gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, [0], toy_handles, fast=fast)
        assert ei.value.kind == "InvalidArgument"
        return
    cuts = np.sort(rng.integers(0, reads.n_reads + 1, n_blocks - 1))
    bf = np.concatenate([[0], cuts, [reads.n_reads]]).astype(np.uint32)
    prefix = rng.integers(0, 40, n_blocks).astype(np.uint32)
    expect = expected_blocks(O, toy_models, reads, bf, fast=fast)
    out, block_off, crc, stats = gctx.compress_blocks(reads.read_off, reads.acids, reads.quals, bf, toy_handles, fast=fast,
                                                      prefix_len=prefix)
    want = [0]
    for b, (data, _, _) in enumerate(expect):
        want.append(want[-1] + 8 + int(prefix[b]) + len(data))
    assert block_off.tolist() == want and stats["out_bytes"] == want[-1]
    check_blocks(out, block_off, crc, expect, prefix)

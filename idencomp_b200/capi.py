"""ctypes binding of the C-ABI in include/idn_gpu.h (libidn_gpu.so).

This is the same surface a Rust ``extern "C"`` block would bind (INTEGRATION.md); Python is used here
because it is what the test and benchmark harness of this repository runs.  There is NO CPU fallback: if the
shared library is missing, or no CUDA device is usable, every call raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libidn_gpu.so"

OK = 0
ERRORS = {
    0: "Ok", 1: "InvalidState", 2: "IoError", 3: "SerializeError", 4: "SequenceTooLong", 5: "InvalidVersion",
    6: "BlockChecksumMismatch", 7: "InvalidModelIndex", 8: "NoActiveModel", 9: "UnknownModel", 10: "Unsupported",
    11: "NoSpace", 12: "InvalidArgument", 13: "InvalidSymbol", 100: "CudaError",
}
MODEL_ACID, MODEL_QSCORE = 0, 1
SPEC_GENERIC, SPEC_LIGHT = 0, 1
MODE_COMPAT, MODE_NATIVE = 1, 2

# every symbol include/idn_gpu.h declares (tests check the library exports all of them)
EXPORTS = [
    "idn_gpu_abi_version", "idn_gpu_device_count", "idn_gpu_create", "idn_gpu_destroy", "idn_gpu_last_error",
    "idn_gpu_launch_count", "idn_gpu_kernel_variant", "idn_gpu_kernel_variant_count", "idn_gpu_set_pipeline_blocks", "idn_gpu_host_alloc", "idn_gpu_host_free", "idn_gpu_model_upload", "idn_gpu_model_release", "idn_gpu_score", "idn_gpu_score_dev",
    "idn_gpu_compress_blocks", "idn_gpu_compress_blocks_dev", "idn_gpu_compress_bound", "idn_gpu_index_blocks",
    "idn_gpu_decompress_blocks", "idn_gpu_decompress_blocks_dev", "idn_gpu_decompress_reads", "idn_gpu_block_crc",
    "idn_gpu_synth_reads_dev", "idn_gpu_profile", "idn_gpu_profile_read", "idn_gpu_set_lane_symbols", "idn_gpu_set_walk",
    "idn_gpu_fastq_parse", "idn_gpu_fastq_parse_dev", "idn_gpu_fastq_fetch", "idn_gpu_fastq_batch_dev", "idn_gpu_fastq_format",
    "idn_gpu_fastq_format_dev", "idn_gpu_fastq_parse_chunk", "idn_gpu_fastq_chunk_fetch", "idn_gpu_compress_parsed",
    "idn_gpu_decompress_to_fastq", "idn_gpu_compress_parsed_ids", "idn_gpu_deflate_names", "idn_gpu_deflate_names_dev",
    "idn_gpu_deflate_names_bound", "idn_gpu_inflate_names", "idn_gpu_inflate_names_fetch", "idn_gpu_set_inflate_range",
    "idn_gpu_decompress_blocks_ids", "idn_gpu_decompress_to_fastq_ids",
]


class IdnGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERRORS.get(code, code)}: {msg}")
        self.code = code
        self.kind = ERRORS.get(code, str(code))


class Batch(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("n_symbols", C.c_uint64), ("n_blocks", C.c_uint32),
                ("acids", C.c_void_p), ("quals", C.c_void_p), ("read_off", C.c_void_p),
                ("block_first_read", C.c_void_p), ("names", C.c_void_p), ("name_off", C.c_void_p)]


class CompressStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("out_bytes", "acid_switches", "q_switches", "payload_bytes", "required_bytes")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class IndexTotals(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("n_symbols", C.c_uint64)]


class FastqInfo(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("n_symbols", C.c_uint64), ("n_name_bytes", C.c_uint64), ("n_lines", C.c_uint64),
                ("error_kind", C.c_int32), ("reserved", C.c_int32), ("bad_record", C.c_uint64)]


class FastqChunk(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("n_symbols", C.c_uint64), ("n_name_bytes", C.c_uint64), ("n_blocks", C.c_uint32),
                ("error_kind", C.c_int32), ("bad_record", C.c_uint64), ("consumed_text", C.c_uint64)]


class InflateStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_streams", "n_chunks", "n_speculative", "n_joined", "serial_bytes", "in_bytes")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


FASTQ_ERRORS = {1: "InvalidFormat", 2: "InvalidAcid", 3: "InvalidQualityScore", 4: "AcidAndQualityScoreLengthMismatch",
                5: "EofReached"}


class ReadIndex(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("pay_off", C.c_void_p), ("pay_len", C.c_void_p), ("seq_len", C.c_void_p),
                ("out_off", C.c_void_p), ("acid_model", C.c_void_p), ("q_model", C.c_void_p)]


_LIB = None


def load():
    """Load libidn_gpu.so and declare prototypes.  Raises if the library has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not LIB_PATH.exists():
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
    L = C.CDLL(str(LIB_PATH))
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int32
    L.idn_gpu_abi_version.restype = i32
    L.idn_gpu_device_count.restype = i32
    L.idn_gpu_create.argtypes = [i32, C.POINTER(vp)]
    L.idn_gpu_create.restype = i32
    L.idn_gpu_destroy.argtypes = [vp]
    L.idn_gpu_destroy.restype = None
    L.idn_gpu_last_error.argtypes = [vp]
    L.idn_gpu_last_error.restype = C.c_char_p
    L.idn_gpu_launch_count.argtypes = [vp]
    L.idn_gpu_launch_count.restype = u64
    L.idn_gpu_kernel_variant.argtypes = [vp, i32, i32]
    L.idn_gpu_kernel_variant.restype = i32
    L.idn_gpu_kernel_variant_count.restype = i32
    L.idn_gpu_host_alloc.argtypes = [u64, C.POINTER(vp)]
    L.idn_gpu_host_alloc.restype = i32
    L.idn_gpu_host_free.argtypes = [vp]
    L.idn_gpu_host_free.restype = None
    L.idn_gpu_set_pipeline_blocks.argtypes = [vp, u32]
    L.idn_gpu_set_pipeline_blocks.restype = i32
    L.idn_gpu_model_upload.argtypes = [vp, i32, i32, i32, i32, i32, i32, u32, vp, vp, vp, u64, C.POINTER(i32)]
    L.idn_gpu_model_upload.restype = i32
    L.idn_gpu_model_release.argtypes = [vp, i32]
    L.idn_gpu_model_release.restype = i32
    L.idn_gpu_score.argtypes = [vp, C.POINTER(Batch), vp, u32, vp]
    L.idn_gpu_score.restype = i32
    L.idn_gpu_score_dev.argtypes = [vp, C.POINTER(Batch), vp, u32, vp, vp]
    L.idn_gpu_score_dev.restype = i32
    L.idn_gpu_compress_blocks.argtypes = [vp, C.POINTER(Batch), i32, vp, u32, i32, vp, vp, u64, vp, vp,
                                          C.POINTER(CompressStats)]
    L.idn_gpu_compress_blocks.restype = i32
    L.idn_gpu_compress_blocks_dev.argtypes = [vp, C.POINTER(Batch), i32, vp, u32, i32, vp, vp, u64, vp, vp, vp, vp]
    L.idn_gpu_compress_blocks_dev.restype = i32
    L.idn_gpu_compress_bound.argtypes = [u64, u64, u32, u64]
    L.idn_gpu_compress_bound.restype = u64
    L.idn_gpu_index_blocks.argtypes = [vp, vp, vp, vp, u32, i32, vp, u32, C.POINTER(IndexTotals), vp]
    L.idn_gpu_index_blocks.restype = i32
    L.idn_gpu_decompress_blocks.argtypes = [vp, vp, vp, vp, vp, u32, i32, vp, u32, vp, vp, vp, vp, vp, u64, u64,
                                            C.POINTER(i32)]
    L.idn_gpu_decompress_blocks.restype = i32
    L.idn_gpu_decompress_blocks_dev.argtypes = [vp, vp, vp, vp, vp, u32, u64, i32, vp, u32, vp, vp, vp, u64, u64, vp, vp]
    L.idn_gpu_decompress_blocks_dev.restype = i32
    L.idn_gpu_decompress_reads.argtypes = [vp, vp, u64, C.POINTER(ReadIndex), vp, u32, vp, vp, vp]
    L.idn_gpu_decompress_reads.restype = i32
    L.idn_gpu_block_crc.argtypes = [vp, C.POINTER(Batch), vp]
    L.idn_gpu_block_crc.restype = i32
    L.idn_gpu_synth_reads_dev.argtypes = [vp, i32, i32, vp, u64, u64, u64, u32, vp, vp, vp]
    L.idn_gpu_synth_reads_dev.restype = i32
    L.idn_gpu_fastq_parse.argtypes = [vp, vp, u64, C.POINTER(FastqInfo)]
    L.idn_gpu_fastq_parse.restype = i32
    L.idn_gpu_fastq_parse_dev.argtypes = [vp, vp, u64, C.POINTER(FastqInfo), vp]
    L.idn_gpu_fastq_parse_dev.restype = i32
    L.idn_gpu_fastq_fetch.argtypes = [vp, vp, vp, vp, vp, vp]
    L.idn_gpu_fastq_fetch.restype = i32
    L.idn_gpu_fastq_batch_dev.argtypes = [vp, C.POINTER(Batch)]
    L.idn_gpu_fastq_batch_dev.restype = i32
    L.idn_gpu_fastq_format.argtypes = [vp, C.POINTER(Batch), i32, vp, u64, C.POINTER(u64)]
    L.idn_gpu_fastq_format.restype = i32
    L.idn_gpu_fastq_format_dev.argtypes = [vp, C.POINTER(Batch), i32, vp, u64, vp, vp]
    L.idn_gpu_fastq_format_dev.restype = i32
    L.idn_gpu_fastq_parse_chunk.argtypes = [vp, vp, u64, i32, u32, C.POINTER(FastqChunk)]
    L.idn_gpu_fastq_parse_chunk.restype = i32
    L.idn_gpu_fastq_chunk_fetch.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.idn_gpu_fastq_chunk_fetch.restype = i32
    L.idn_gpu_compress_parsed.argtypes = [vp, i32, vp, u32, i32, i32, vp, vp, u64, vp, vp, C.POINTER(CompressStats)]
    L.idn_gpu_compress_parsed.restype = i32
    L.idn_gpu_decompress_to_fastq.argtypes = [vp, vp, vp, vp, vp, u32, i32, vp, u32, vp, vp, u64, u64, i32, vp, u64, C.POINTER(u64),
                                             C.POINTER(u64), C.POINTER(i32)]
    L.idn_gpu_decompress_to_fastq.restype = i32
    L.idn_gpu_compress_parsed_ids.argtypes = [vp, i32, vp, u32, i32, vp, u64, vp, vp, C.POINTER(CompressStats)]
    L.idn_gpu_compress_parsed_ids.restype = i32
    L.idn_gpu_deflate_names.argtypes = [vp, vp, vp, vp, u32, vp, u64, vp]
    L.idn_gpu_deflate_names.restype = i32
    L.idn_gpu_deflate_names_dev.argtypes = [vp, vp, vp, vp, u32, vp, u64, vp, vp]
    L.idn_gpu_deflate_names_dev.restype = i32
    L.idn_gpu_deflate_names_bound.argtypes = [u64, u64, u32]
    L.idn_gpu_deflate_names_bound.restype = u64
    L.idn_gpu_inflate_names.argtypes = [vp, vp, vp, vp, u32, vp, u64, C.POINTER(u64), C.POINTER(i32), C.POINTER(InflateStats)]
    L.idn_gpu_inflate_names.restype = i32
    L.idn_gpu_inflate_names_fetch.argtypes = [vp, vp, vp]
    L.idn_gpu_inflate_names_fetch.restype = i32
    L.idn_gpu_set_inflate_range.argtypes = [vp, u32]
    L.idn_gpu_set_inflate_range.restype = i32
    L.idn_gpu_decompress_blocks_ids.argtypes = [vp, vp, vp, vp, vp, u32, i32, vp, u32, vp, vp, vp, u64, u64, C.POINTER(i32)]
    L.idn_gpu_decompress_blocks_ids.restype = i32
    L.idn_gpu_decompress_to_fastq_ids.argtypes = [vp, vp, vp, vp, vp, u32, i32, vp, u32, u64, u64, i32, vp, u64, C.POINTER(u64),
                                                  C.POINTER(u64), C.POINTER(i32)]
    L.idn_gpu_decompress_to_fastq_ids.restype = i32
    L.idn_gpu_set_lane_symbols.argtypes = [vp, u32]
    L.idn_gpu_set_lane_symbols.restype = i32
    L.idn_gpu_set_walk.argtypes = [vp, i32]
    L.idn_gpu_set_walk.restype = i32
    L.idn_gpu_profile.argtypes = [vp, i32]
    L.idn_gpu_profile.restype = i32
    L.idn_gpu_profile_read.argtypes = [vp, C.c_char_p, u64]
    L.idn_gpu_profile_read.restype = i32
    _LIB = L
    return L


def _p(a):
    if a is None:
        return None
    return a.ctypes.data if a.size else None


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def make_batch(read_off, acids, quals, block_first_read=None, name_off=None, names=None):
    """Host idn_batch from numpy arrays; returns (Batch, keepalive)."""
    ro = _c(read_off, np.uint64)
    a = _c(acids, np.uint8)
    q = _c(quals, np.uint8)
    n_reads = len(ro) - 1
    if block_first_read is None:
        block_first_read = [0, n_reads]
    bf = _c(block_first_read, np.uint32)
    b = Batch()
    b.n_reads = n_reads
    b.n_symbols = int(ro[-1]) if len(ro) else 0
    b.n_blocks = len(bf) - 1
    b.acids, b.quals = _p(a), _p(q)
    b.read_off = ro.ctypes.data
    b.block_first_read = bf.ctypes.data
    keep = [ro, a, q, bf]
    if name_off is not None:
        no = _c(name_off, np.uint64)
        nm = _c(names, np.uint8)
        if nm.size == 0:
            nm = np.zeros(1, dtype=np.uint8)
        b.name_off = no.ctypes.data
        b.names = nm.ctypes.data
        keep += [no, nm]
    return b, keep


class Context:
    """idn_gpu_ctx: one per device per host thread."""

    def __init__(self, device: int = 0):
        self.L = load()
        h = C.c_void_p()
        rc = self.L.idn_gpu_create(device, C.byref(h))
        if rc != OK:
            raise IdnGpuError(rc, f"idn_gpu_create(device={device}) failed: no usable CUDA device (no CPU fallback)")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.idn_gpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int):
        if rc != OK:
            raise IdnGpuError(rc, self.L.idn_gpu_last_error(self.h).decode())

    @property
    def launches(self) -> int:
        return int(self.L.idn_gpu_launch_count(self.h))

    def kernel_variant(self, acid_handle: int, q_handle: int) -> int:
        """index of the compile-time-specialised codec kernels this pair launches, -1 = the run-time-generic ones"""
        return int(self.L.idn_gpu_kernel_variant(self.h, acid_handle, q_handle))

    def set_pipeline_blocks(self, n: int):
        """blocks per sub-chunk of the pipelined host-pointer calls (include/idn_gpu.h)"""
        self.check(self.L.idn_gpu_set_pipeline_blocks(self.h, n))

    def set_lane_symbols(self, n: int):
        self.check(self.L.idn_gpu_set_lane_symbols(self.h, n))

    def set_walk(self, mode: int):
        """0 automatic, 1 one-warp-per-block slice walk, 2 parallel speculative walk first (include/idn_gpu.h)"""
        self.check(self.L.idn_gpu_set_walk(self.h, mode))

    def profile(self, enable: bool):
        self.check(self.L.idn_gpu_profile(self.h, int(enable)))

    def profile_read(self) -> dict:
        """{kernel: (launches, total_ms)} since the last read."""
        buf = C.create_string_buffer(1 << 16)
        self.check(self.L.idn_gpu_profile_read(self.h, buf, len(buf)))
        out = {}
        for ln in buf.value.decode().splitlines():
            name, n, ms = ln.split()
            out[name] = (int(n), float(ms))
        return out

    # ---- models -------------------------------------------------------------------------------
    def upload_model(self, mtype: int, kind: int, ao: int, qo: int, pb: int, qmax: int, cum, spec_keys, spec_ctx) -> int:
        cum = _c(cum, np.uint16)
        keys = _c(spec_keys, np.uint32)
        ctx = _c(spec_ctx, np.uint32)
        n_ctx = cum.shape[0] - 1
        h = C.c_int32(-1)
        self.check(self.L.idn_gpu_model_upload(self.h, mtype, kind, ao, qo, pb, qmax, n_ctx, cum.ctypes.data,
                                               _p(keys), _p(ctx), len(keys), C.byref(h)))
        return int(h.value)

    def release_model(self, handle: int):
        self.check(self.L.idn_gpu_model_release(self.h, handle))

    # ---- host-pointer entry points ------------------------------------------------------------------
    def score(self, batch_arrays, models) -> np.ndarray:
        b, keep = make_batch(*batch_arrays)
        m = _c(models, np.int32)
        sizes = np.zeros((b.n_reads, len(m)), dtype=np.uint32)
        self.check(self.L.idn_gpu_score(self.h, C.byref(b), _p(m), len(m), _p(sizes)))
        return sizes

    def deflate_names(self, name_off, names, block_first_read, *, out_cap=None):
        """identifiers slices (0x00 | u32be n | 0x01 | raw Deflate of the block's names joined by '\\n') of every block,
        Deflated on the device -> (slices, slice_off[n_blocks + 1])"""
        no = _c(name_off, np.uint64)
        nm = _c(names, np.uint8)
        if nm.size == 0:
            nm = np.zeros(1, dtype=np.uint8)
        bf = _c(block_first_read, np.uint32)
        nb = len(bf) - 1
        if out_cap is None:
            out_cap = int(self.L.idn_gpu_deflate_names_bound(int(no[-1] - no[0]), len(no) - 1, nb))
        out = np.zeros(max(out_cap, 1), dtype=np.uint8)
        so = np.zeros(nb + 1, dtype=np.uint64)
        rc = self.L.idn_gpu_deflate_names(self.h, nm.ctypes.data, no.ctypes.data, bf.ctypes.data, nb, out.ctypes.data, out_cap, so.ctypes.data)
        if rc != OK:
            e = IdnGpuError(rc, self.L.idn_gpu_last_error(self.h).decode())
            e.required = int(so[-1])
            raise e
        return out[:int(so[-1])], so

    def set_inflate_range(self, n: int):
        """compressed bytes per range of the parallel inflate (idn_gpu_set_inflate_range)"""
        self.check(self.L.idn_gpu_set_inflate_range(self.h, n))

    def inflate_names(self, blocks, block_off, block_first_read, *, block_len=None, resident=False):
        """the blocks' Identifiers slices inflated and split into names on the device -> (names, name_off, stats).
        blocks: payloads as idn_gpu_decompress_blocks takes them; resident=True passes blocks == NULL (the bytes of the last
        index_blocks call).  A failure raises IdnGpuError with .bad_block and .stats."""
        bo = _c(block_off, np.uint64)
        bl = None if block_len is None else _c(block_len, np.uint32)
        bf = _c(block_first_read, np.uint32)
        blk = None if resident else _c(blocks, np.uint8)
        if blk is not None and blk.size == 0:
            blk = np.zeros(1, dtype=np.uint8)
        n_reads = int(bf[-1])
        nb, bad, st = C.c_uint64(0), C.c_int32(-1), InflateStats()
        rc = self.L.idn_gpu_inflate_names(self.h, _p(blk), bo.ctypes.data, _p(bl), len(bo) - 1, bf.ctypes.data, n_reads, C.byref(nb),
                                          C.byref(bad), C.byref(st))
        if rc != OK:
            e = IdnGpuError(rc, self.L.idn_gpu_last_error(self.h).decode())
            e.bad_block = int(bad.value)
            e.stats = st.as_dict()
            raise e
        names = np.zeros(max(1, nb.value), dtype=np.uint8)
        name_off = np.zeros(n_reads + 1, dtype=np.uint64)
        self.check(self.L.idn_gpu_inflate_names_fetch(self.h, names.ctypes.data, name_off.ctypes.data))
        return names[:nb.value], name_off, st.as_dict()

    def compress_blocks(self, read_off, acids, quals, block_first_read, models, *, fast=False, prefix_len=None,
                        name_off=None, names=None, out_cap=None, mode=MODE_COMPAT):
        b, keep = make_batch(read_off, acids, quals, block_first_read, name_off, names)
        m = _c(models, np.int32)
        pl = None if prefix_len is None else _c(prefix_len, np.uint32)
        ptot = 0 if pl is None else int(pl.sum())
        if out_cap is None:
            out_cap = int(self.L.idn_gpu_compress_bound(b.n_reads, b.n_symbols, b.n_blocks, ptot))
        out = np.zeros(max(out_cap, 1), dtype=np.uint8)
        block_off = np.zeros(b.n_blocks + 1, dtype=np.uint64)
        crc = np.zeros(max(b.n_blocks, 1), dtype=np.uint32)
        st = CompressStats()
        rc = self.L.idn_gpu_compress_blocks(self.h, C.byref(b), mode, _p(m), len(m), int(fast), _p(pl), out.ctypes.data,
                                            out_cap, block_off.ctypes.data, crc.ctypes.data, C.byref(st))
        if rc != OK:
            e = IdnGpuError(rc, self.L.idn_gpu_last_error(self.h).decode())
            e.stats = st.as_dict()
            raise e
        return out[:st.out_bytes], block_off, crc[:b.n_blocks], st.as_dict()

    def index_blocks(self, blocks, block_off, models, block_len=None, mode=MODE_COMPAT):
        blocks = _c(blocks, np.uint8)
        bo = _c(block_off, np.uint64)
        bl = None if block_len is None else _c(block_len, np.uint32)
        m = _c(models, np.int32)
        tot = IndexTotals()
        bf = np.zeros(len(bo), dtype=np.uint32)
        self.check(self.L.idn_gpu_index_blocks(self.h, _p(blocks), bo.ctypes.data, _p(bl), len(bo) - 1, mode, _p(m), len(m),
                                               C.byref(tot), bf.ctypes.data))
        return int(tot.n_reads), int(tot.n_symbols), bf

    def decompress_blocks(self, blocks, block_off, block_crc, models, *, name_off=None, names=None, reads_cap=None,
                          symbols_cap=None, mode=MODE_COMPAT, block_len=None, resident=False):
        """resident=True: index the blocks, then decode the bytes that call left on the device (blocks == NULL)"""
        blocks = _c(blocks, np.uint8)
        bo = _c(block_off, np.uint64)
        bl = None if block_len is None else _c(block_len, np.uint32)
        m = _c(models, np.int32)
        nb = len(bo) - 1
        if reads_cap is None or symbols_cap is None:
            reads_cap, symbols_cap, _ = self.index_blocks(blocks, bo, m, bl, mode)
        crc = None if block_crc is None else _c(block_crc, np.uint32)
        a = np.zeros(max(symbols_cap, 1), dtype=np.uint8)
        q = np.zeros(max(symbols_cap, 1), dtype=np.uint8)
        ro = np.zeros(reads_cap + 1, dtype=np.uint64)
        bad = C.c_int32(-1)
        no = nm = None
        if name_off is not None:
            no = _c(name_off, np.uint64)
            nm = _c(names, np.uint8)
            if nm.size == 0:
                nm = np.zeros(1, dtype=np.uint8)
        if resident:
            reads_cap, symbols_cap, _ = self.index_blocks(blocks, bo, m, bl, mode)
        rc = self.L.idn_gpu_decompress_blocks(self.h, None if resident else _p(blocks), bo.ctypes.data, _p(bl), _p(crc), nb, mode, _p(m), len(m),
                                              None if nm is None else nm.ctypes.data,
                                              None if no is None else no.ctypes.data, a.ctypes.data, q.ctypes.data,
                                              ro.ctypes.data, reads_cap, symbols_cap, C.byref(bad))
        if rc != OK:
            e = IdnGpuError(rc, self.L.idn_gpu_last_error(self.h).decode())
            e.bad_block = int(bad.value)
            raise e
        n = int(ro[-1]) if reads_cap else 0
        return ro, a[:n], q[:n]

    def decompress_reads(self, payload, pay_off, pay_len, seq_len, acid_model, q_model, models, out_off=None):
        """Decode reads from their payloads (idn_read_index).  out_off defaults to the exclusive scan of seq_len.  On error
        the raised IdnGpuError carries .read_status (the per-read status the kernel wrote; zeros if it never ran)."""
        payload = _c(payload, np.uint8)
        po = _c(pay_off, np.uint64)
        pl = _c(pay_len, np.uint32)
        sl = _c(seq_len, np.uint32)
        am = _c(acid_model, np.uint8)
        qm = _c(q_model, np.uint8)
        m = _c(models, np.int32)
        if out_off is None:
            oo = np.zeros(len(sl) + 1, dtype=np.uint64)
            np.cumsum(sl, out=oo[1:])
        else:
            oo = _c(out_off, np.uint64)
        idx = ReadIndex(len(sl), _p(po), _p(pl), _p(sl), oo.ctypes.data, _p(am), _p(qm))
        S = int(sl.sum(dtype=np.uint64))
        a = np.zeros(max(S, 1), dtype=np.uint8)
        q = np.zeros(max(S, 1), dtype=np.uint8)
        st = np.zeros(max(len(sl), 1), dtype=np.uint32)
        rc = self.L.idn_gpu_decompress_reads(self.h, _p(payload), payload.size, C.byref(idx), _p(m), len(m),
                                             a.ctypes.data, q.ctypes.data, st.ctypes.data)
        if rc != OK:
            e = IdnGpuError(rc, self.L.idn_gpu_last_error(self.h).decode())
            e.read_status = st[:len(sl)]
            raise e
        return oo, a[:S], q[:S], st[:len(sl)]

    def block_crc(self, read_off, acids, quals, block_first_read, name_off=None, names=None) -> np.ndarray:
        b, keep = make_batch(read_off, acids, quals, block_first_read, name_off, names)
        crc = np.zeros(max(b.n_blocks, 1), dtype=np.uint32)
        self.check(self.L.idn_gpu_block_crc(self.h, C.byref(b), crc.ctypes.data))
        return crc[:b.n_blocks]

    # ---- FASTQ text <-> symbols (row f1) ------------------------------------------------------------------
    def fastq_parse(self, text: bytes):
        """FastqReader over a whole buffer -> (read_off, acids, quals, name_off, names).  Raises IdnGpuError
        (SerializeError) with .fastq_error / .bad_record on malformed input."""
        buf = np.frombuffer(text, dtype=np.uint8)
        info = FastqInfo()
        rc = self.L.idn_gpu_fastq_parse(self.h, buf.ctypes.data if buf.size else None, buf.size, C.byref(info))
        if rc != OK:
            e = IdnGpuError(rc, self.L.idn_gpu_last_error(self.h).decode())
            e.fastq_error = FASTQ_ERRORS.get(int(info.error_kind), str(info.error_kind))
            e.bad_record = int(info.bad_record)
            raise e
        a = np.zeros(max(info.n_symbols, 1), dtype=np.uint8)
        q = np.zeros(max(info.n_symbols, 1), dtype=np.uint8)
        ro = np.zeros(info.n_reads + 1, dtype=np.uint64)
        nm = np.zeros(max(info.n_name_bytes, 1), dtype=np.uint8)
        no = np.zeros(info.n_reads + 1, dtype=np.uint64)
        self.check(self.L.idn_gpu_fastq_fetch(self.h, a.ctypes.data, q.ctypes.data, ro.ctypes.data, nm.ctypes.data, no.ctypes.data))
        return ro, a[:info.n_symbols], q[:info.n_symbols], no, nm[:info.n_name_bytes]

    def fastq_format(self, read_off, acids, quals, name_off=None, names=None, title_with_separator=False) -> bytes:
        """FastqWriter::write_sequence for every read."""
        b, keep = make_batch(read_off, acids, quals, None, name_off, names)
        n_reads, S = b.n_reads, b.n_symbols
        nb = 0 if name_off is None else int(np.asarray(name_off)[-1])
        cap = 2 * S + 6 * n_reads + nb * (2 if title_with_separator else 1) + 16
        out = np.zeros(cap, dtype=np.uint8)
        n = C.c_uint64(0)
        self.check(self.L.idn_gpu_fastq_format(self.h, C.byref(b), int(title_with_separator), out.ctypes.data, cap, C.byref(n)))
        return out[:n.value].tobytes()

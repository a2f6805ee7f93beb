"""ctypes binding of the CPU oracle (oracle/liboracle.so).

TEST INFRASTRUCTURE ONLY -- see oracle/idn_oracle.h.  Only tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / ``--impl reference`` legs may import this module; the product package
(idencomp_b200/) never does.

Model files are read here with the Python ``msgpack`` package and the identifier is recomputed with
``hashlib.sha3_256`` -- an implementation independent of the product's own C++ msgpack/SHA3 loader, so
the two check each other (reference: model_serializer.rs:66-72,177-189; model.rs:458-482).
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import re
import struct
import subprocess
from dataclasses import dataclass
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB = None

ACID, QSCORE = 0, 1
NSYM = {ACID: 5, QSCORE: 94}
ERRORS = {
    0: "Ok", 1: "InvalidState", 2: "IoError", 3: "SerializeError", 4: "SequenceTooLong",
    5: "InvalidVersion", 6: "BlockChecksumMismatch", 7: "InvalidModelIndex", 8: "NoActiveModel",
    9: "UnknownModel", 10: "Unsupported", 11: "FastqError",
}


class OracleError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERRORS.get(code, code)}: {msg}")
        self.code = code
        self.kind = ERRORS.get(code, str(code))


def build(force: bool = False) -> Path:
    so = _HERE / "liboracle.so"
    src = [_HERE / "idn_oracle.c", _HERE / "idn_oracle.h"]
    if force or not so.exists() or any(s.stat().st_mtime > so.stat().st_mtime for s in src):
        subprocess.run(["make", "-C", str(_HERE), "-s", "-B", "liboracle.so"], check=True)
    return so


class _Spec(C.Structure):
    _fields_ = [("kind", C.c_int), ("ao", C.c_int), ("qo", C.c_int), ("pb", C.c_int), ("qmax", C.c_int)]


class _Gen(C.Structure):
    _fields_ = [("spec", _Spec)] + [(n, C.c_uint32) for n in (
        "base_a", "base_q", "abits", "qbits", "last_pow_a", "last_pow_q", "astate", "qstate",
        "position", "length")]


class _Params(C.Structure):
    _fields_ = [("models", C.POINTER(C.c_void_p)), ("n_models", C.c_uint32),
                ("max_block_total_len", C.c_uint32), ("include_identifiers", C.c_int),
                ("quality", C.c_int), ("fast", C.c_int), ("threads", C.c_int), ("deflate_level", C.c_int)]


class _Reads(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("total_len", C.c_uint64), ("read_off", C.c_void_p),
                ("acids", C.c_void_p), ("quals", C.c_void_p), ("name_off", C.c_void_p),
                ("names", C.c_void_p)]


class _Buf(C.Structure):
    _fields_ = [("data", C.c_void_p), ("len", C.c_size_t), ("cap", C.c_size_t)]


class _Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_blocks", "acid_switches", "q_switches", "out_acid_bytes",
                                          "out_q_score_bytes", "names_bytes")]


class _Decoded(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("total_len", C.c_uint64), ("read_off", C.c_void_p),
                ("acids", C.c_void_p), ("quals", C.c_void_p), ("name_off", C.c_void_p),
                ("names", C.c_void_p), ("version", C.c_uint8), ("n_models", C.c_uint32),
                ("model_ids", (C.c_uint8 * 32) * 256), ("n_blocks", C.c_uint64)]


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(str(build()))
        L.orc_last_error.restype = C.c_char_p
        L.orc_model_new.restype = C.c_void_p
        L.orc_model_new.argtypes = [C.c_int, C.c_char_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_size_t, C.c_void_p]
        L.orc_model_free.argtypes = [C.c_void_p]
        L.orc_model_cum_row.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        L.orc_model_ctx_for.argtypes = [C.c_void_p, C.c_uint32]
        L.orc_model_ctx_for.restype = C.c_uint32
        L.orc_quantise.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.orc_spec_parse.argtypes = [C.c_char_p, C.POINTER(_Spec)]
        L.orc_spec_num.argtypes = [C.POINTER(_Spec)]
        L.orc_spec_num.restype = C.c_uint64
        L.orc_gen_init.argtypes = [C.POINTER(_Gen), C.POINTER(_Spec), C.c_uint32]
        L.orc_gen_current.argtypes = [C.POINTER(_Gen)]
        L.orc_gen_current.restype = C.c_uint32
        L.orc_gen_update.argtypes = [C.POINTER(_Gen), C.c_uint8, C.c_uint8]
        L.orc_encode_read.restype = C.c_size_t
        L.orc_encode_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        L.orc_decode_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_score_read.restype = C.c_size_t
        L.orc_score_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
        L.orc_rans_encode_raw.restype = C.c_size_t
        L.orc_rans_encode_raw.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p]
        L.orc_compress.argtypes = [C.POINTER(_Params), C.POINTER(_Reads), C.POINTER(_Buf), C.POINTER(_Stats)]
        L.orc_compress_block.argtypes = [C.POINTER(_Params), C.POINTER(_Reads), C.c_uint64, C.c_uint64,
                                         C.POINTER(_Buf), C.POINTER(C.c_uint32), C.POINTER(_Stats)]
        L.orc_decompress.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_void_p, C.c_size_t, C.c_int,
                                     C.POINTER(_Decoded)]
        L.orc_fastq_parse.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(_Decoded)]
        L.orc_fastq_write.argtypes = [C.POINTER(_Reads), C.POINTER(_Buf)]
        L.orc_buf_free.argtypes = [C.POINTER(_Buf)]
        L.orc_decoded_free.argtypes = [C.POINTER(_Decoded)]
        L.orc_compress_native_block.argtypes = [C.POINTER(_Params), C.POINTER(_Reads), C.c_uint64, C.c_uint64, C.c_uint32,
                                                C.POINTER(_Buf), C.POINTER(C.c_uint32)]
        L.orc_native_block_counts.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.orc_decompress_native_block.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_void_p, C.c_size_t, C.c_void_p,
                                                  C.c_void_p, C.c_void_p]
        L.orc_synth_reads.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32,
                                      C.c_int, C.c_void_p, C.c_void_p]
        L.orc_crc32.restype = C.c_uint32
        L.orc_crc32.argtypes = [C.c_uint32, C.c_void_p, C.c_size_t]
        _LIB = L
    return _LIB


def _check(rc: int):
    if rc != 0:
        raise OracleError(rc, lib().orc_last_error().decode())


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


# ---------------------------------------------------------------------------------------------
# primitives
# ---------------------------------------------------------------------------------------------
def quantise(probs, scale_bits: int = 14) -> np.ndarray:
    p = np.ascontiguousarray(probs, dtype=np.float32)
    out = np.zeros(len(p), dtype=np.uint32)
    lib().orc_quantise(_ptr(p), len(p), scale_bits, _ptr(out))
    return out


def spec_num(name: str) -> int:
    s = _Spec()
    if lib().orc_spec_parse(name.encode(), C.byref(s)) != 0:
        raise ValueError(f"bad spec type {name}")
    return int(lib().orc_spec_num(C.byref(s)))


class Generator:
    """ContextSpecGenerator (context_spec.rs:186-214)."""

    def __init__(self, name: str, length: int):
        s = _Spec()
        if lib().orc_spec_parse(name.encode(), C.byref(s)) != 0:
            raise ValueError(f"bad spec type {name}")
        self._g = _Gen()
        lib().orc_gen_init(C.byref(self._g), C.byref(s), length)

    def current_context(self) -> int:
        return int(lib().orc_gen_current(C.byref(self._g)))

    def update(self, acid: int, q: int) -> None:
        lib().orc_gen_update(C.byref(self._g), acid, q)


def rans_encode_raw(starts, freqs, nstates: int, scale_bits: int) -> bytes:
    s = np.ascontiguousarray(starts, dtype=np.uint32)
    f = np.ascontiguousarray(freqs, dtype=np.uint32)
    out = np.zeros(2 * len(s) + 4 * nstates, dtype=np.uint8)
    n = lib().orc_rans_encode_raw(_ptr(s), _ptr(f), len(s), nstates, scale_bits, _ptr(out))
    return out[:n].tobytes()


def crc32(data, crc: int = 0) -> int:
    a = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data)
    return int(lib().orc_crc32(crc, _ptr(a), a.size))


# ---------------------------------------------------------------------------------------------
# models
# ---------------------------------------------------------------------------------------------
def make_identifier(mtype: int, spec_name: str, probs: np.ndarray, keys: np.ndarray, ctx: np.ndarray) -> bytes:
    """Model::make_identifier (model.rs:458-482)."""
    h = hashlib.sha3_256()
    h.update(bytes([mtype]))
    h.update(spec_name.encode())
    h.update(np.ascontiguousarray(probs, dtype=">f4").tobytes())
    order = np.argsort(keys, kind="stable")
    pairs = np.empty((len(keys), 2), dtype=">u4")
    pairs[:, 0] = np.asarray(keys)[order]
    pairs[:, 1] = np.asarray(ctx)[order]
    h.update(pairs.tobytes())
    return h.digest()


@dataclass
class ModelData:
    """Plain arrays of a model: what both the oracle and the product's C-ABI consume."""
    mtype: int
    spec_name: str
    probs: np.ndarray      # [n_ctx, nsym] f32
    spec_keys: np.ndarray  # [n_specs] u32
    spec_ctx: np.ndarray   # [n_specs] u32 (0-based context index)
    identifier: bytes

    @property
    def n_ctx(self) -> int:
        return int(self.probs.shape[0])

    @staticmethod
    def from_contexts(mtype: int, spec_name: str, contexts) -> "ModelData":
        """Model::with_model_and_spec_type (model.rs:216-249): contexts = [(specs, probs)], sorted by specs."""
        contexts = sorted(contexts, key=lambda c: list(c[0]))
        nsym = NSYM[mtype]
        probs = np.zeros((len(contexts), nsym), dtype=np.float32)
        keys, ctx = [], []
        for i, (specs, p) in enumerate(contexts):
            probs[i] = np.asarray(p, dtype=np.float32)
            keys.extend(specs)
            ctx.extend([i] * len(specs))
        keys = np.asarray(keys, dtype=np.uint32)
        ctx = np.asarray(ctx, dtype=np.uint32)
        return ModelData(mtype, spec_name, probs, keys, ctx, make_identifier(mtype, spec_name, probs, keys, ctx))

    @staticmethod
    def empty(mtype: int) -> "ModelData":
        """Model::empty (model.rs:251-259)."""
        return ModelData.from_contexts(mtype, "dummy", [])

    @staticmethod
    def load_msgpack(path) -> "ModelData":
        """SerializableModel::read_model (model_serializer.rs:66-72, 111-114, 177-189)."""
        import msgpack
        ident, mtype_s, spec_name, ctxs = msgpack.unpackb(Path(path).read_bytes(), raw=False)
        mtype = {"Acids": ACID, "QualityScores": QSCORE}[mtype_s]
        md = ModelData.from_contexts(mtype, spec_name, [(c[0], c[1][1]) for c in ctxs])
        if md.identifier != bytes(ident):
            raise ValueError(f"{path}: identifier mismatch")
        return md


class Model:
    """RansEncModel + RansDecModel of one model (sequence_compressor.rs:12-48,167-205)."""

    def __init__(self, md: ModelData):
        self.md = md
        probs = np.ascontiguousarray(md.probs, dtype=np.float32)
        keys = np.ascontiguousarray(md.spec_keys, dtype=np.uint32)
        ctx = np.ascontiguousarray(md.spec_ctx, dtype=np.uint32)
        ident = np.frombuffer(md.identifier, dtype=np.uint8)
        self.h = lib().orc_model_new(md.mtype, md.spec_name.encode(), md.n_ctx, _ptr(probs), _ptr(keys),
                                     _ptr(ctx), len(keys), _ptr(ident))
        if not self.h:
            raise ValueError("orc_model_new failed (bad spec type or > 65536 contexts)")

    def __del__(self):
        if getattr(self, "h", None) and _LIB is not None:
            _LIB.orc_model_free(self.h)
            self.h = None

    @property
    def mtype(self) -> int:
        return self.md.mtype

    def cum_row(self, ctx: int) -> np.ndarray:
        out = np.zeros(NSYM[self.md.mtype] + 1, dtype=np.uint32)
        lib().orc_model_cum_row(self.h, ctx, _ptr(out))
        return out

    def cum_table(self) -> np.ndarray:
        """[(n_ctx+1), nsym+1] u16, row 0 = dummy, last column = 16384."""
        n = self.md.n_ctx + 1
        return np.stack([self.cum_row(i) for i in range(n)]).astype(np.uint16)

    def ctx_for(self, spec: int) -> int:
        return int(lib().orc_model_ctx_for(self.h, spec))


# ---------------------------------------------------------------------------------------------
# per-read codec
# ---------------------------------------------------------------------------------------------
def encode_read(am: Model, qm: Model, acids: np.ndarray, quals: np.ndarray) -> bytes:
    a = np.ascontiguousarray(acids, dtype=np.uint8)
    q = np.ascontiguousarray(quals, dtype=np.uint8)
    out = np.zeros(4 * len(a) + 8, dtype=np.uint8)
    n = lib().orc_encode_read(am.h, qm.h, _ptr(a), _ptr(q), len(a), _ptr(out))
    return out[:n].tobytes()


def decode_read(am: Model, qm: Model, data: bytes, seq_len: int):
    d = np.frombuffer(data, dtype=np.uint8)
    a = np.zeros(max(seq_len, 1), dtype=np.uint8)
    q = np.zeros(max(seq_len, 1), dtype=np.uint8)
    st = np.zeros(2, dtype=np.uint32)
    used = C.c_size_t(0)
    _check(lib().orc_decode_read(am.h, qm.h, _ptr(d), len(d), seq_len, _ptr(a), _ptr(q), _ptr(st), C.byref(used)))
    return a[:seq_len], q[:seq_len], (int(st[0]), int(st[1])), int(used.value)


def score_read(m: Model, acids: np.ndarray, quals: np.ndarray) -> int:
    a = np.ascontiguousarray(acids, dtype=np.uint8)
    q = np.ascontiguousarray(quals, dtype=np.uint8)
    return int(lib().orc_score_read(m.h, _ptr(a), _ptr(q), len(a)))


# ---------------------------------------------------------------------------------------------
# reads container + whole-file API
# ---------------------------------------------------------------------------------------------
@dataclass
class Reads:
    """SoA batch of FASTQ records: the layout the C-ABI boundary uses (SURVEY.md 8b)."""
    read_off: np.ndarray  # [R+1] u64
    acids: np.ndarray     # [sum len] u8 0..4
    quals: np.ndarray     # [sum len] u8 0..93
    name_off: np.ndarray | None = None  # [R+1] u64
    names: np.ndarray | None = None     # u8

    @property
    def n_reads(self) -> int:
        return len(self.read_off) - 1

    def name(self, r: int) -> bytes:
        if self.name_off is None:
            return b""
        return self.names[self.name_off[r]:self.name_off[r + 1]].tobytes()

    def _c(self) -> _Reads:
        self.read_off = np.ascontiguousarray(self.read_off, dtype=np.uint64)
        self.acids = np.ascontiguousarray(self.acids, dtype=np.uint8)
        self.quals = np.ascontiguousarray(self.quals, dtype=np.uint8)
        r = _Reads()
        r.n_reads = self.n_reads
        r.total_len = int(self.read_off[-1])
        r.read_off = self.read_off.ctypes.data
        r.acids = self.acids.ctypes.data if self.acids.size else None
        r.quals = self.quals.ctypes.data if self.quals.size else None
        if self.name_off is not None:
            self.name_off = np.ascontiguousarray(self.name_off, dtype=np.uint64)
            self.names = np.ascontiguousarray(self.names, dtype=np.uint8)
            r.name_off = self.name_off.ctypes.data
            r.names = self.names.ctypes.data if self.names.size else None
        return r

    def without_names(self) -> "Reads":
        return Reads(self.read_off, self.acids, self.quals, None, None)

    @staticmethod
    def from_lists(seqs) -> "Reads":
        """seqs = [(name: bytes|str, acids, quals)]"""
        ro, no = [0], [0]
        a, q, n = [], [], []
        for name, ac, qu in seqs:
            if isinstance(name, str):
                name = name.encode()
            a.append(np.asarray(ac, dtype=np.uint8))
            q.append(np.asarray(qu, dtype=np.uint8))
            n.append(np.frombuffer(name, dtype=np.uint8))
            ro.append(ro[-1] + len(ac))
            no.append(no[-1] + len(name))
        cat = lambda xs: np.concatenate(xs) if xs else np.zeros(0, dtype=np.uint8)
        return Reads(np.asarray(ro, dtype=np.uint64), cat(a), cat(q), np.asarray(no, dtype=np.uint64), cat(n))


def _take_decoded(d: _Decoded) -> Reads:
    R, T = int(d.n_reads), int(d.total_len)

    def arr(p, n, dt):
        if n == 0 or not p:
            return np.zeros(0, dtype=dt)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n * np.dtype(dt).itemsize,)).view(dt).copy()

    ro = arr(d.read_off, R + 1, np.uint64)
    no = arr(d.name_off, R + 1, np.uint64)
    out = Reads(ro, arr(d.acids, T, np.uint8), arr(d.quals, T, np.uint8), no,
                arr(d.names, int(no[-1]) if len(no) else 0, np.uint8))
    return out


def fastq_parse(text: bytes) -> Reads:
    """FastqReader::read_sequence until EOF (fastq/reader.rs:166-282).  On malformed input raises OracleError
    (FastqError) with .fastq_error = the FastqReaderError variant (as capi.FASTQ_ERRORS names it) and .bad_record =
    the 0-based record, in file order, that the reference stops at."""
    t = np.frombuffer(text, dtype=np.uint8)
    d = _Decoded()
    rc = lib().orc_fastq_parse(_ptr(t), len(t), C.byref(d))
    if rc != 0:
        msg = lib().orc_last_error().decode()
        e = OracleError(rc, msg)
        m = re.fullmatch(r"FastqReaderError::(\w+) at record (\d+)", msg)
        if m is None:
            raise e
        e.fastq_error, e.bad_record = m.group(1), int(m.group(2))
        raise e
    try:
        return _take_decoded(d)
    finally:
        lib().orc_decoded_free(C.byref(d))


def fastq_write(reads: Reads) -> bytes:
    b = _Buf()
    _check(lib().orc_fastq_write(C.byref(reads._c()), C.byref(b)))
    try:
        return C.string_at(b.data, b.len) if b.len else b""
    finally:
        lib().orc_buf_free(C.byref(b))


def _params(models, max_block_total_len, include_identifiers, quality, fast, threads):
    arr = (C.c_void_p * len(models))(*[m.h for m in models])
    p = _Params()
    p.models = C.cast(arr, C.POINTER(C.c_void_p))
    p.n_models = len(models)
    p.max_block_total_len = max_block_total_len
    p.include_identifiers = int(include_identifiers)
    p.quality = 1 if fast else quality
    p.fast = int(fast)
    p.threads = threads
    p.deflate_level = 6
    return p, arr


def compress(models, reads: Reads, *, max_block_total_len: int = 4 * 1024 * 1024,
             include_identifiers: bool = True, quality: int = 7, fast: bool = False, threads: int = 0,
             return_stats: bool = False):
    """IdnCompressor::with_params + add_sequence* + finish (idn/compressor.rs:443-585)."""
    p, keep = _params(models, max_block_total_len, include_identifiers, quality, fast, threads)
    b, st = _Buf(), _Stats()
    rd = reads if include_identifiers else reads.without_names()
    _check(lib().orc_compress(C.byref(p), C.byref(rd._c()), C.byref(b), C.byref(st)))
    try:
        data = C.string_at(b.data, b.len)
    finally:
        lib().orc_buf_free(C.byref(b))
    if return_stats:
        return data, {n: int(getattr(st, n)) for n, _ in _Stats._fields_}
    return data


def compress_block(models, reads: Reads, first: int, n: int, *, include_identifiers=True, quality=7, fast=False):
    p, keep = _params(models, 0, include_identifiers, quality, fast, 0)
    b, st = _Buf(), _Stats()
    crc = C.c_uint32(0)
    rd = reads if include_identifiers else reads.without_names()
    _check(lib().orc_compress_block(C.byref(p), C.byref(rd._c()), first, n, C.byref(b), C.byref(crc), C.byref(st)))
    try:
        data = C.string_at(b.data, b.len) if b.len else b""
    finally:
        lib().orc_buf_free(C.byref(b))
    return data, int(crc.value), {n_: int(getattr(st, n_)) for n_, _ in _Stats._fields_}


# ---- GPU-native multi-lane format (container version 2, DESIGN.md section 8): our own format, stated independently ----
def compress_native_block(models, reads: Reads, first: int, n: int, *, lane_syms: int = 4096, include_identifiers=True,
                          fast=False):
    """Slices of one version-2 block (no block header) and its CRC."""
    p, keep = _params(models, 0, include_identifiers, 7, fast, 0)
    b = _Buf()
    crc = C.c_uint32(0)
    rd = reads if include_identifiers else reads.without_names()
    _check(lib().orc_compress_native_block(C.byref(p), C.byref(rd._c()), first, n, lane_syms, C.byref(b), C.byref(crc)))
    try:
        data = C.string_at(b.data, b.len) if b.len else b""
    finally:
        lib().orc_buf_free(C.byref(b))
    return data, int(crc.value)


def decompress_native_block(models, data: bytes):
    """(read_len[], acids, quals) of one version-2 block's slices."""
    buf = np.frombuffer(data, dtype=np.uint8)
    nr, ns = C.c_uint64(0), C.c_uint64(0)
    _check(lib().orc_native_block_counts(_ptr(buf), len(buf), C.byref(nr), C.byref(ns)))
    a = np.zeros(max(ns.value, 1), dtype=np.uint8)
    q = np.zeros(max(ns.value, 1), dtype=np.uint8)
    ln = np.zeros(max(nr.value, 1), dtype=np.uint32)
    arr = (C.c_void_p * max(len(models), 1))(*[m.h for m in models])
    _check(lib().orc_decompress_native_block(C.cast(arr, C.POINTER(C.c_void_p)), len(models), _ptr(buf), len(buf),
                                             a.ctypes.data, q.ctypes.data, ln.ctypes.data))
    return ln[:nr.value], a[:ns.value], q[:ns.value]


def decompress(models, idn: bytes, threads: int = 0, return_info: bool = False):
    """IdnDecompressor::with_params + next_sequence* (idn/decompressor.rs:455-566)."""
    arr = (C.c_void_p * max(len(models), 1))(*[m.h for m in models])
    d = _Decoded()
    buf = np.frombuffer(idn, dtype=np.uint8)
    _check(lib().orc_decompress(C.cast(arr, C.POINTER(C.c_void_p)), len(models), _ptr(buf), len(buf), threads, C.byref(d)))
    try:
        reads = _take_decoded(d)
        info = {"n_blocks": int(d.n_blocks), "n_models": int(d.n_models),
                "model_ids": [bytes(d.model_ids[i]) for i in range(int(d.n_models))]}
    finally:
        lib().orc_decoded_free(C.byref(d))
    return (reads, info) if return_info else reads


# ---------------------------------------------------------------------------------------------
# the reference's toy models (_internal_test_data.rs:245-304), rebuilt from their definitions
# ---------------------------------------------------------------------------------------------
def synth_reads(am: "Model", qm: "Model", read_off, first_read_index: int, seed: int, n_ppm: int,
                threads: int = 0) -> "Reads":
    """Model-driven synthetic reads (bench/test utility, SURVEY.md 8d); same sampler as idn_gpu_synth_reads_dev."""
    ro = np.ascontiguousarray(read_off, dtype=np.uint64)
    n = int(ro[-1])
    a = np.zeros(max(n, 1), dtype=np.uint8)
    q = np.zeros(max(n, 1), dtype=np.uint8)
    _check(lib().orc_synth_reads(am.h, qm.h, ro.ctypes.data, len(ro) - 1, first_read_index, seed, n_ppm, threads,
                                 a.ctypes.data, q.ctypes.data))
    return Reads(ro, a[:n], q[:n], None, None)


def simple_acid_model() -> ModelData:
    """create_simple_acid_model (_internal_test_data.rs:245-262): generic_ao1_qo0_pb0, specs = acid value."""
    ctxs = [([1], [0.00, 0.80, 0.10, 0.05, 0.05]), ([2], [0.00, 0.25, 0.50, 0.15, 0.10]),
            ([3], [0.00, 0.01, 0.01, 0.97, 0.01]), ([4], [0.00, 0.30, 0.30, 0.30, 0.10])]
    return ModelData.from_contexts(ACID, "generic_ao1_qo0_pb0", ctxs)


def simple_q_score_model() -> ModelData:
    """create_simple_qscore_model (_internal_test_data.rs:286-304): generic_ao0_qo1_pb0."""
    ctxs = []
    for i in range(94):
        p = [0.06 if i == j else 0.01 for j in range(94)]
        ctxs.append(([i], p))
    return ModelData.from_contexts(QSCORE, "generic_ao0_qo1_pb0", ctxs)


def acid_model_prefer(sym: int) -> ModelData:
    """create_acid_model_prefer_a / _c (_internal_test_data.rs:264-284): Dummy spec type, 1 context."""
    p = [0.001, 0.033, 0.033, 0.033, 0.033]
    p[sym] = 0.900
    return ModelData.from_contexts(ACID, "dummy", [([0], p)])

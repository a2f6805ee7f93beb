"""ctypes binding of include/idn_host.h (libidn_host.so): the C++ host mirror of idencomp's API.

Model loading (msgpack + SHA3 identifier check + bit-exact f32 quantiser) happens in the C++ library; Python only
passes paths and pointers.  No CPU codec lives here: everything that touches symbols goes to libidn_gpu.so.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from . import capi

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libidn_host.so"

EXPORTS = [
    "idn_host_last_error", "idn_host_model_load", "idn_host_model_from_bytes", "idn_host_model_new",
    "idn_host_model_empty", "idn_host_model_free", "idn_host_model_type", "idn_host_model_len",
    "idn_host_model_spec_name", "idn_host_model_identifier", "idn_host_model_cum_table", "idn_host_model_upload",
    "idn_host_quantise", "idn_host_params_default", "idn_host_compressor_new", "idn_host_compressor_add",
    "idn_host_compressor_add_batch", "idn_host_compressor_finish", "idn_host_compressor_output",
    "idn_host_compressor_retained", "idn_host_compressor_stats", "idn_host_compressor_free", "idn_host_decompress",
    "idn_host_decoded_reads", "idn_host_decoded_version", "idn_host_decoded_read_off", "idn_host_decoded_acids",
    "idn_host_decoded_quals", "idn_host_decoded_name_off", "idn_host_decoded_names", "idn_host_decoded_free",
    "idn_host_cluster", "idn_host_rank", "idn_host_clustering_new", "idn_host_clustering_free", "idn_host_splitmix64",
    "idn_host_xoshiro256pp", "idn_host_sample_indices", "idn_host_gen_range", "idn_host_compressor_add_text", "idn_host_decompress_text",
    "idn_host_text_free", "idn_host_decompress_text_into", "idn_host_compressor_set_output",
    "idn_host_release_cached", "idn_host_text_reader_new", "idn_host_text_reader_next", "idn_host_text_reader_free",
    "idn_host_decompress_ex", "idn_host_decompress_text_ex", "idn_host_decompress_text_into_ex", "idn_host_text_reader_new_ex",
]


class DecompressParams(C.Structure):
    """idn_host_decompress_params: the IdnDecompressorParams the _ex entry points take"""
    _fields_ = [("identifiers_on_device", C.c_int32)]


def _dparams(identifiers_on_device: bool):
    return C.byref(DecompressParams(int(bool(identifiers_on_device))))


class Params(C.Structure):
    """idn_host_params = IdnCompressorParamsBuilder (idn/compressor.rs:164-274) + device / mode / batching."""
    _fields_ = [("max_block_total_len", C.c_uint32), ("thread_num", C.c_uint32), ("include_identifiers", C.c_int32),
                ("quality", C.c_uint32), ("fast", C.c_int32), ("device", C.c_int32), ("mode", C.c_int32),
                ("batch_blocks", C.c_uint32), ("lane_symbols", C.c_uint32), ("text_chunk_bytes", C.c_uint64), ("n_devices", C.c_uint32),
                ("devices", C.c_int32 * 16), ("identifiers_on_device", C.c_int32)]

_LIB = None


def load():
    global _LIB
    if _LIB is not None:
        return _LIB
    capi.load()
    if not LIB_PATH.exists():
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    L = C.CDLL(str(LIB_PATH))
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int32
    L.idn_host_last_error.restype = C.c_char_p
    L.idn_host_model_load.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.idn_host_model_from_bytes.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
    L.idn_host_model_new.argtypes = [i32, C.c_char_p, u32, vp, vp, vp, u64, C.POINTER(vp)]
    L.idn_host_model_empty.argtypes = [i32, C.POINTER(vp)]
    L.idn_host_model_free.argtypes = [vp]
    L.idn_host_model_free.restype = None
    L.idn_host_model_type.argtypes = [vp]
    L.idn_host_model_len.argtypes = [vp]
    L.idn_host_model_len.restype = u32
    L.idn_host_model_spec_name.argtypes = [vp]
    L.idn_host_model_spec_name.restype = C.c_char_p
    L.idn_host_model_identifier.argtypes = [vp, vp]
    L.idn_host_model_identifier.restype = None
    L.idn_host_model_cum_table.argtypes = [vp, vp, u64]
    L.idn_host_model_cum_table.restype = u64
    L.idn_host_model_upload.argtypes = [vp, vp, C.POINTER(i32)]
    L.idn_host_quantise.argtypes = [vp, u32, u32, vp]
    L.idn_host_params_default.argtypes = [C.POINTER(Params)]
    L.idn_host_params_default.restype = None
    L.idn_host_compressor_new.argtypes = [vp, u32, C.POINTER(Params), C.POINTER(vp)]
    L.idn_host_compressor_add.argtypes = [vp, vp, u64, vp, vp, u64]
    L.idn_host_compressor_add_batch.argtypes = [vp, u64, vp, vp, vp, vp, vp]
    L.idn_host_compressor_add_text.argtypes = [vp, vp, u64]
    L.idn_host_decompress_text.argtypes = [vp, u32, i32, u32, u32, i32, vp, u64, C.POINTER(vp), C.POINTER(u64)]
    L.idn_host_decompress_text_into.argtypes = [vp, u32, i32, u32, u32, i32, vp, u64, vp, u64, C.POINTER(u64)]
    L.idn_host_compressor_set_output.argtypes = [vp, vp, u64]
    L.idn_host_text_reader_new.argtypes = [vp, u32, C.POINTER(i32), u32, u32, u32, i32, vp, u64, C.POINTER(vp)]
    L.idn_host_text_reader_next.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    L.idn_host_text_reader_free.argtypes = [vp]
    L.idn_host_text_reader_free.restype = None
    L.idn_host_release_cached.argtypes = []
    L.idn_host_release_cached.restype = None
    L.idn_host_text_free.argtypes = [vp]
    L.idn_host_text_free.restype = None
    L.idn_host_compressor_finish.argtypes = [vp]
    L.idn_host_compressor_output.argtypes = [vp, C.POINTER(vp)]
    L.idn_host_compressor_output.restype = u64
    L.idn_host_compressor_retained.argtypes = [vp, vp, u32]
    L.idn_host_compressor_retained.restype = u32
    L.idn_host_compressor_stats.argtypes = [vp, vp]
    L.idn_host_compressor_stats.restype = None
    L.idn_host_compressor_free.argtypes = [vp]
    L.idn_host_compressor_free.restype = None
    L.idn_host_decompress.argtypes = [vp, u32, i32, u32, vp, u64, C.POINTER(vp)]
    L.idn_host_decompress_ex.argtypes = [vp, u32, i32, u32, vp, u64, C.POINTER(vp), C.POINTER(DecompressParams)]
    L.idn_host_decompress_text_ex.argtypes = [vp, u32, i32, u32, u32, i32, vp, u64, C.POINTER(vp), C.POINTER(u64), C.POINTER(DecompressParams)]
    L.idn_host_decompress_text_into_ex.argtypes = [vp, u32, i32, u32, u32, i32, vp, u64, vp, u64, C.POINTER(u64), C.POINTER(DecompressParams)]
    L.idn_host_text_reader_new_ex.argtypes = [vp, u32, C.POINTER(i32), u32, u32, u32, i32, vp, u64, C.POINTER(vp),
                                              C.POINTER(DecompressParams)]
    for name, rt in (("reads", u64), ("version", u32), ("read_off", vp), ("acids", vp), ("quals", vp), ("name_off", vp), ("names", vp)):
        f = getattr(L, "idn_host_decoded_" + name)
        f.argtypes = [vp]
        f.restype = rt
    L.idn_host_decoded_free.argtypes = [vp]
    L.idn_host_decoded_free.restype = None
    L.idn_host_clustering_new.argtypes = []
    L.idn_host_clustering_new.restype = vp
    L.idn_host_clustering_free.argtypes = [vp]
    L.idn_host_clustering_free.restype = None
    L.idn_host_cluster.argtypes = [vp, vp, u64, u32, u32, vp, vp]
    L.idn_host_cluster.restype = u32
    L.idn_host_splitmix64.argtypes = [u64, u32, vp]
    L.idn_host_splitmix64.restype = None
    L.idn_host_xoshiro256pp.argtypes = [vp, u64, u32, vp]
    L.idn_host_xoshiro256pp.restype = None
    L.idn_host_sample_indices.argtypes = [u64, u32, u32, vp]
    L.idn_host_sample_indices.restype = u32
    L.idn_host_gen_range.argtypes = [u64, u32, u32, vp]
    L.idn_host_gen_range.restype = u32
    L.idn_host_rank.argtypes = [vp, u64, u32, u32, vp]
    L.idn_host_rank.restype = u32
    _LIB = L
    return L


class HostError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{capi.ERRORS.get(code, code)}: {msg}")
        self.code = code
        self.kind = capi.ERRORS.get(code, str(code))


def _check(rc: int):
    if rc != 0:
        raise HostError(rc, load().idn_host_last_error().decode())


def quantise(probs, scale_bits: int = 14) -> np.ndarray:
    """Context::as_integer_cum_freqs (context.rs:346-371)."""
    p = np.ascontiguousarray(probs, dtype=np.float32)
    out = np.zeros(len(p), dtype=np.uint32)
    _check(load().idn_host_quantise(p.ctypes.data, len(p), scale_bits, out.ctypes.data))
    return out


class Model:
    """idencomp::Model (model.rs:176-259)."""

    def __init__(self, handle):
        self.L = load()
        self.h = handle

    @staticmethod
    def load(path) -> "Model":
        h = C.c_void_p()
        _check(load().idn_host_model_load(str(path).encode(), C.byref(h)))
        return Model(h)

    @staticmethod
    def from_bytes(data: bytes) -> "Model":
        h = C.c_void_p()
        buf = np.frombuffer(data, dtype=np.uint8)
        _check(load().idn_host_model_from_bytes(buf.ctypes.data, len(buf), C.byref(h)))
        return Model(h)

    @staticmethod
    def new(model_type: int, spec_name: str, probs, spec_keys, spec_ctx) -> "Model":
        p = np.ascontiguousarray(probs, dtype=np.float32)
        k = np.ascontiguousarray(spec_keys, dtype=np.uint32)
        c = np.ascontiguousarray(spec_ctx, dtype=np.uint32)
        h = C.c_void_p()
        _check(load().idn_host_model_new(model_type, spec_name.encode(), p.shape[0] if p.ndim == 2 else 0,
                                         p.ctypes.data if p.size else None, k.ctypes.data if k.size else None,
                                         c.ctypes.data if c.size else None, len(k), C.byref(h)))
        return Model(h)

    @staticmethod
    def empty(model_type: int) -> "Model":
        h = C.c_void_p()
        _check(load().idn_host_model_empty(model_type, C.byref(h)))
        return Model(h)

    def __del__(self):
        try:
            if self.h:
                self.L.idn_host_model_free(self.h)
                self.h = None
        except Exception:
            pass

    @property
    def model_type(self) -> int:
        return int(self.L.idn_host_model_type(self.h))

    def __len__(self) -> int:
        return int(self.L.idn_host_model_len(self.h))

    @property
    def spec_name(self) -> str:
        return self.L.idn_host_model_spec_name(self.h).decode()

    @property
    def identifier(self) -> bytes:
        out = (C.c_uint8 * 32)()
        self.L.idn_host_model_identifier(self.h, out)
        return bytes(out)

    def cum_table(self) -> np.ndarray:
        nsym = 5 if self.model_type == 0 else 94
        out = np.zeros((len(self) + 1, nsym + 1), dtype=np.uint16)
        self.L.idn_host_model_cum_table(self.h, out.ctypes.data, out.size)
        return out

    def upload(self, ctx: "capi.Context") -> int:
        """RansEncModel/RansDecModel::from_model on the device; returns the idn_model_t handle."""
        h = C.c_int32(-1)
        _check(self.L.idn_host_model_upload(ctx.h, self.h, C.byref(h)))
        return int(h.value)


def _model_array(models):
    arr = (C.c_void_p * max(len(models), 1))(*[m.h for m in models])
    return arr


class IdnCompressor:
    """idencomp::IdnCompressor (idn/compressor.rs:443-585) writing to memory.

        c = IdnCompressor(models, quality=7, include_identifiers=True)   # IdnCompressor::with_params
        identifiers_on_device=True: the identifiers slices are Deflated on the GPU instead of by the host's zlib
        c.add_sequence(b"name", acids, quals) ; ... ; idn = c.finish()
    """

    def __init__(self, models, *, max_block_total_len=4 * 1024 * 1024, thread_num=0, include_identifiers=True, quality=7,
                 fast=False, device=0, devices=None, mode=capi.MODE_COMPAT, batch_blocks=32, lane_symbols=2048, text_chunk_bytes=0,
                 identifiers_on_device=False):
        self.L = load()
        p = Params()
        self.L.idn_host_params_default(C.byref(p))
        p.max_block_total_len, p.thread_num, p.include_identifiers = max_block_total_len, thread_num, int(include_identifiers)
        p.quality, p.fast, p.device, p.mode, p.batch_blocks, p.lane_symbols = quality, int(fast), device, mode, batch_blocks, lane_symbols
        if text_chunk_bytes:
            p.text_chunk_bytes = text_chunk_bytes
        p.identifiers_on_device = int(identifiers_on_device)
        if devices:  # several GPUs share the file: same container, whatever their number
            p.n_devices = len(devices)
            for i, d in enumerate(devices):
                p.devices[i] = d
        self._models = list(models)
        h = C.c_void_p()
        _check(self.L.idn_host_compressor_new(_model_array(self._models), len(self._models), C.byref(p), C.byref(h)))
        self.h = h

    def add_sequence(self, name: bytes, acids, quals):
        a = np.ascontiguousarray(acids, dtype=np.uint8)
        q = np.ascontiguousarray(quals, dtype=np.uint8)
        if len(a) != len(q):
            raise ValueError("acids and quality scores differ in length")
        nm = np.frombuffer(name, dtype=np.uint8) if name else np.zeros(0, dtype=np.uint8)
        _check(self.L.idn_host_compressor_add(self.h, nm.ctypes.data if nm.size else None, nm.size,
                                              a.ctypes.data if a.size else None, q.ctypes.data if q.size else None, len(a)))

    def add_batch(self, read_off, acids, quals, name_off=None, names=None):
        ro = np.ascontiguousarray(read_off, dtype=np.uint64)
        a = np.ascontiguousarray(acids, dtype=np.uint8)
        q = np.ascontiguousarray(quals, dtype=np.uint8)
        no = nm = None
        if name_off is not None:
            no = np.ascontiguousarray(name_off, dtype=np.uint64)
            nm = np.ascontiguousarray(names, dtype=np.uint8)
            if nm.size == 0:
                nm = np.zeros(1, dtype=np.uint8)
        _check(self.L.idn_host_compressor_add_batch(self.h, len(ro) - 1, ro.ctypes.data, a.ctypes.data if a.size else None,
                                                    q.ctypes.data if q.size else None, None if no is None else no.ctypes.data,
                                                    None if nm is None else nm.ctypes.data))

    def set_output(self, buf: np.ndarray):
        """write the container into `buf` (a uint8 array, e.g. page-locked) instead of the library's growing buffer"""
        self._out_keep = buf
        _check(self.L.idn_host_compressor_set_output(self.h, buf.ctypes.data, buf.size))

    def add_fastq_text(self, text):
        """consecutive pieces of FASTQ text, cut anywhere (bytes or a uint8 array; not to be mixed with add_sequence / add_batch)"""
        buf = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray, memoryview)) else np.ascontiguousarray(text, dtype=np.uint8)
        _check(self.L.idn_host_compressor_add_text(self.h, buf.ctypes.data if buf.size else None, buf.size))

    def finish(self, copy: bool = True):
        """copy=False: no bytes object of the container is made (read it with output_view() or from the set_output buffer)"""
        _check(self.L.idn_host_compressor_finish(self.h))
        return self.output() if copy else None

    def output_view(self) -> np.ndarray:
        """the container written so far as a uint8 view of the library's buffer (valid until the next call on this object)"""
        ptr = C.c_void_p()
        n = self.L.idn_host_compressor_output(self.h, C.byref(ptr))
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), (n,)) if n else np.zeros(0, dtype=np.uint8)

    def output(self) -> bytes:
        ptr = C.c_void_p()
        n = self.L.idn_host_compressor_output(self.h, C.byref(ptr))
        return C.string_at(ptr, n) if n else b""

    def retained_models(self):
        buf = (C.c_uint8 * (32 * 255))()
        n = self.L.idn_host_compressor_retained(self.h, buf, 255)
        return [bytes(buf[32 * i:32 * i + 32]) for i in range(n)]

    def stats(self) -> dict:
        out = (C.c_uint64 * 9)()
        self.L.idn_host_compressor_stats(self.h, out)
        keys = ("in_symbols", "in_reads", "in_identifier_bytes", "out_bytes", "out_identifier_bytes", "out_payload_bytes",
                "blocks", "acid_model_switches", "q_score_model_switches")
        return dict(zip(keys, (int(v) for v in out)))

    def close(self):
        if getattr(self, "h", None):
            self.L.idn_host_compressor_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def decompress(models, idn: bytes, *, device=0, n_devices=0, batch_blocks=32, identifiers_on_device=False) -> dict:
    """idencomp::IdnDecompressor (idn/decompressor.rs:455-566): every sequence of the file as one SoA batch.
    n_devices > 1: the first n_devices GPUs share the file.  identifiers_on_device: the Identifiers slices are inflated on
    the device (Brotli slices still on the host); the result does not change."""
    if n_devices > 1:
        device = -n_devices
    L = load()
    buf = np.frombuffer(idn, dtype=np.uint8)
    h = C.c_void_p()
    models = list(models)
    _check(L.idn_host_decompress_ex(_model_array(models), len(models), device, batch_blocks, buf.ctypes.data if buf.size else None,
                                    buf.size, C.byref(h), _dparams(identifiers_on_device)))
    try:
        n = int(L.idn_host_decoded_reads(h))
        ro = np.ctypeslib.as_array(C.cast(L.idn_host_decoded_read_off(h), C.POINTER(C.c_uint64)), (n + 1,)).copy()
        no = np.ctypeslib.as_array(C.cast(L.idn_host_decoded_name_off(h), C.POINTER(C.c_uint64)), (n + 1,)).copy()
        S, NB = int(ro[-1]), int(no[-1])
        take = lambda p, k: np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), (k,)).copy() if k else np.zeros(0, dtype=np.uint8)
        return {"version": int(L.idn_host_decoded_version(h)), "read_off": ro, "acids": take(L.idn_host_decoded_acids(h), S),
                "quals": take(L.idn_host_decoded_quals(h), S), "name_off": no, "names": take(L.idn_host_decoded_names(h), NB)}
    finally:
        L.idn_host_decoded_free(h)


def decompress_text(models, idn, *, device=0, n_devices=0, batch_blocks=32, thread_num=0, title_with_separator=False, as_view=False,
                    identifiers_on_device=False):
    """IdnDecompressor + FastqWriter (fastq/writer.rs:190-245): the whole file as FASTQ text, formatted on the device.
    identifiers_on_device: the names are inflated on the device too and never cross to the host."""
    L = load()
    buf = np.frombuffer(idn, dtype=np.uint8) if isinstance(idn, (bytes, bytearray, memoryview)) else np.ascontiguousarray(idn, dtype=np.uint8)
    models = list(models)
    if n_devices > 1:
        device = -n_devices
    ptr, n = C.c_void_p(), C.c_uint64(0)
    _check(L.idn_host_decompress_text_ex(_model_array(models), len(models), device, batch_blocks, thread_num, int(title_with_separator),
                                         buf.ctypes.data if buf.size else None, buf.size, C.byref(ptr), C.byref(n),
                                         _dparams(identifiers_on_device)))
    if as_view:  # (view, free): no copy of the text; call free() when done with the view
        view = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), (n.value,)) if n.value else np.zeros(0, dtype=np.uint8)
        return view, (lambda: L.idn_host_text_free(ptr))
    try:
        return C.string_at(ptr, n.value) if n.value else b""
    finally:
        L.idn_host_text_free(ptr)


def decompress_text_into(models, idn, out: np.ndarray, *, device=0, n_devices=0, batch_blocks=32, thread_num=0, title_with_separator=False,
                         identifiers_on_device=False) -> int:
    """decompress_text into the caller's uint8 array (e.g. page-locked); returns the length of the text"""
    L = load()
    buf = np.frombuffer(idn, dtype=np.uint8) if isinstance(idn, (bytes, bytearray, memoryview)) else np.ascontiguousarray(idn, dtype=np.uint8)
    models = list(models)
    if n_devices > 1:
        device = -n_devices
    n = C.c_uint64(0)
    _check(L.idn_host_decompress_text_into_ex(_model_array(models), len(models), device, batch_blocks, thread_num, int(title_with_separator),
                                              buf.ctypes.data if buf.size else None, buf.size, out.ctypes.data, out.size, C.byref(n),
                                              _dparams(identifiers_on_device)))
    return int(n.value)


def release_cached():
    """give back the device contexts and page-locked buffers the library keeps between compressors / decompressors"""
    load().idn_host_release_cached()


class FastqTextReader:
    """streaming text out: iterating yields the FASTQ text of one batch of blocks at a time as a uint8 view of the library's
    page-locked memory (valid until the next step) -- what a writer would hand to write()"""

    def __init__(self, models, idn, *, devices=(0,), batch_blocks=32, thread_num=0, title_with_separator=False, identifiers_on_device=False):
        self.L = load()
        self._idn = np.frombuffer(idn, dtype=np.uint8) if isinstance(idn, (bytes, bytearray, memoryview)) else np.ascontiguousarray(idn, dtype=np.uint8)
        models = list(models)
        self._models = models
        devs = (C.c_int32 * max(1, len(devices)))(*devices)
        h = C.c_void_p()
        _check(self.L.idn_host_text_reader_new_ex(_model_array(models), len(models), devs, len(devices), batch_blocks, thread_num,
                                                  int(title_with_separator), self._idn.ctypes.data if self._idn.size else None, self._idn.size,
                                                  C.byref(h), _dparams(identifiers_on_device)))
        self.h = h

    def __iter__(self):
        return self

    def __next__(self):
        p, n = C.c_void_p(), C.c_uint64(0)
        _check(self.L.idn_host_text_reader_next(self.h, C.byref(p), C.byref(n)))
        if n.value == 0:
            raise StopIteration
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n.value,))

    def close(self):
        if self.h:
            self.L.idn_host_text_reader_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Clustering:
    """Clustering (clustering.rs:8-118): one random stream (Xoshiro256++ seeded with 404) that runs on from one
    make_clusters call to the next, as the reference's ModelChooser uses it for the acid and then the q-score models."""

    def __init__(self):
        self.h = load().idn_host_clustering_new()

    def make_clusters(self, cost, num_clusters: int):
        return cluster(cost, num_clusters, self)

    def close(self):
        if self.h:
            load().idn_host_clustering_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def cluster(cost, num_clusters: int, state: "Clustering | None" = None):
    """Clustering::make_clusters (clustering.rs:21-118) on cost[value][centroid] -> (centroids, cluster of every value).
    state = None: a fresh Clustering::new()."""
    c = np.ascontiguousarray(cost, dtype=np.uint32)
    cent = np.zeros(max(num_clusters, 1), dtype=np.uint32)
    vc = np.zeros(max(c.shape[0], 1), dtype=np.uint32)
    n = load().idn_host_cluster(state.h if state else None, c.ctypes.data, c.shape[0], c.shape[1], num_clusters, cent.ctypes.data,
                                vc.ctypes.data)
    return cent[:n].tolist(), vc[:c.shape[0]].tolist()


def splitmix64(seed: int, n: int):
    out = np.zeros(n, dtype=np.uint64)
    load().idn_host_splitmix64(seed, n, out.ctypes.data)
    return out.tolist()


def xoshiro256pp(n: int, *, state=None, seed: int = 0):
    """n outputs of Xoshiro256++ started from four state words, or from seed_from_u64(seed)."""
    out = np.zeros(n, dtype=np.uint64)
    st = None if state is None else np.asarray(state, dtype=np.uint64)
    load().idn_host_xoshiro256pp(None if st is None else st.ctypes.data, seed, n, out.ctypes.data)
    return out.tolist()


def sample_indices(seed: int, length: int, amount: int):
    """rand 0.8.5 index::sample(&mut Xoshiro256PlusPlus::seed_from_u64(seed), length, amount) (amount < 12)."""
    out = np.zeros(max(amount, 1), dtype=np.uint32)
    n = load().idn_host_sample_indices(seed, length, amount, out.ctypes.data)
    return out[:n].tolist()


def gen_range(seed: int, high: int, n: int):
    """n draws of rng.gen_range(0..=high) on Xoshiro256PlusPlus::seed_from_u64(seed)."""
    out = np.zeros(n, dtype=np.uint32)
    load().idn_host_gen_range(seed, high, n, out.ctypes.data)
    return out.tolist()


def rank(cost, model_num: int):
    """get_model_ranking (idn/model_chooser.rs:103-138) on cost[read][model] -> best model columns."""
    c = np.ascontiguousarray(cost, dtype=np.uint32)
    out = np.zeros(max(model_num, 1), dtype=np.uint32)
    n = load().idn_host_rank(c.ctypes.data, c.shape[0], c.shape[1], model_num, out.ctypes.data)
    return out[:n].tolist()

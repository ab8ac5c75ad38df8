"""ctypes access to the CPU checkers (test infrastructure only).

  oracle/libzso.so                 plain-C restatement ("port")
  oracle/_ref/libzstd-oracle.so    the reference's own libzstd 1.5.7, compiled in place by oracle/Makefile
  tests/hostsim/libzb_hostsim.so   1-lane host instantiation of the CUDA kernel source

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.

The ref_* functions answer from the compiled reference when oracle/_ref is built.  Without it they answer from
tests/golden/reference_results.json: what the compiled reference returned for the same call, an error code as such and any
other result as a digest (a Recorded, equal to exactly the bytes / array / list it digests).  To refresh that file, run the
whole suite, GPU tests included, where oracle/_ref is built with ZSTDB200_RECORD_REFERENCE=<file>: every live reference call is
added to <file>.
"""
from __future__ import annotations

import atexit
import ctypes as C
import functools
import hashlib
import inspect
import json
import os
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
ZSO_PATH = ROOT / "oracle" / "libzso.so"
REF_PATH = ROOT / "oracle" / "_ref" / "libzstd-oracle.so"
HOSTSIM_PATH = ROOT / "tests" / "hostsim" / "libzb_hostsim.so"
RESULTS_PATH = ROOT / "tests" / "golden" / "reference_results.json"

ERR_MAX = (1 << 64) - 120
_cache = {}


def digest(x) -> str:
    """48-bit SHA-256 prefix of a result: bytes, a uint32 record array (shape included) or a JSON-able list."""
    if isinstance(x, Recorded):
        return x.digest
    if isinstance(x, (bytes, bytearray)):
        b = bytes(x)
    elif hasattr(x, "dtype"):
        import numpy as np
        b = repr(tuple(x.shape)).encode() + np.ascontiguousarray(x, dtype="<u4").tobytes()
    else:
        b = json.dumps(x).encode()
    return hashlib.sha256(b).hexdigest()[:12]


class Recorded:
    """A non-error result of the compiled reference, known by its digest."""

    def __init__(self, d: str):
        self.digest = d

    def __eq__(self, other):
        return not isinstance(other, int) and digest(other) == self.digest

    __hash__ = None

    def __repr__(self):
        return f"<reference result {self.digest}>"


def same(expected, got) -> bool:
    """expected (a live or Recorded reference result) equals got; arrays compare whole."""
    if isinstance(expected, int) or isinstance(got, int):
        return isinstance(expected, int) and isinstance(got, int) and expected == got
    return digest(expected) == digest(got)


def _call_key(name: str, args) -> str:
    h = hashlib.sha256(name.encode())
    for a in args:
        h.update(hashlib.sha256(a).digest() if isinstance(a, (bytes, bytearray)) else json.dumps(a, sort_keys=True).encode())
        h.update(b"|")
    return h.hexdigest()[:12]


_results = None
_recording = {} if os.environ.get("ZSTDB200_RECORD_REFERENCE") else None


def _save_recording():
    path = Path(os.environ["ZSTDB200_RECORD_REFERENCE"])
    old = json.loads(path.read_text()) if path.exists() else {}
    old.update(_recording)
    path.write_text(json.dumps(dict(sorted(old.items())), indent=0) + "\n")


if _recording is not None:
    atexit.register(_save_recording)


def _recorded(fn):
    """fn runs on the compiled reference when it is built; otherwise the recorded result of the same call is returned."""
    sig = inspect.signature(fn)

    @functools.wraps(fn)
    def call(*args, **kwargs):
        global _results
        bound = sig.bind(*args, **kwargs)
        bound.apply_defaults()
        key = _call_key(fn.__name__, list(bound.arguments.values()))
        if ref() is not None:
            r = fn(*args, **kwargs)
            if _recording is not None:
                _recording[key] = r if isinstance(r, int) else digest(r)
            return r
        if _results is None:
            _results = json.loads(RESULTS_PATH.read_text())
        if key not in _results:
            raise LookupError(f"{fn.__name__}: no recorded reference result for this call in {RESULTS_PATH.name}; record it where oracle/_ref "
                              "is built (ZSTDB200_RECORD_REFERENCE, see the docstring of tests/oracle_util.py)")
        r = _results[key]
        return r if isinstance(r, int) else Recorded(r)
    return call


def _load(path, protos):
    if path in _cache:
        return _cache[path]
    if not Path(path).exists():
        _cache[path] = None
        return None
    L = C.CDLL(str(path))
    for name, res, args in protos:
        f = getattr(L, name)
        f.restype = res
        f.argtypes = args
    _cache[path] = L
    return L


def zso():
    L = _load(ZSO_PATH, [
        ("zso_compress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int]),
        ("zso_compress_flags", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int, C.c_uint]),
        ("zso_decompress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t]),
        ("zso_compressBound", C.c_size_t, [C.c_size_t]),
        ("zso_findFrameCompressedSize", C.c_size_t, [C.c_char_p, C.c_size_t]),
        ("zso_getFrameContentSize", C.c_ulonglong, [C.c_char_p, C.c_size_t]),
    ])
    if L is None:
        raise RuntimeError(f"{ZSO_PATH} missing: run `make -C oracle` (or __graft_entry__.build())")
    return L


def ref():
    """The compiled reference, or None when oracle/_ref was not built (it needs the reference's sources)."""
    return _load(REF_PATH, [
        ("ZSTD_compress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int]),
        ("ZSTD_decompress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t]),
        ("ZSTD_compressBound", C.c_size_t, [C.c_size_t]),
        ("ZSTD_createCCtx", C.c_void_p, []),
        ("ZSTD_freeCCtx", C.c_size_t, [C.c_void_p]),
        ("ZSTD_createDCtx", C.c_void_p, []),
        ("ZSTD_freeDCtx", C.c_size_t, [C.c_void_p]),
        ("ZSTD_CCtx_setParameter", C.c_size_t, [C.c_void_p, C.c_int, C.c_int]),
        ("ZSTD_CCtx_reset", C.c_size_t, [C.c_void_p, C.c_int]),
        ("ZSTD_compress2", C.c_size_t, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
        ("ZSTD_decompressDCtx", C.c_size_t, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
        ("ZSTD_compressStream2", C.c_size_t, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
        ("ZSTD_versionString", C.c_char_p, []),
        ("ZSTD_DCtx_setParameter", C.c_size_t, [C.c_void_p, C.c_int, C.c_int]),
        ("ZSTD_generateSequences", C.c_size_t, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t]),
        ("ZSTD_sequenceBound", C.c_size_t, [C.c_size_t]),
        ("ZSTD_registerSequenceProducer", None, [C.c_void_p, C.c_void_p, C.c_void_p]),
    ])


def hostsim():
    L = _load(HOSTSIM_PATH, [
        ("zbh_compress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int]),
        ("zbh_compress_flags", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int, C.c_uint]),
        ("zbh_decompress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t]),
        ("zbh_decompress_format", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_uint]),
        ("zbh_compress_bound", C.c_size_t, [C.c_size_t]),
        ("zbe_compress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int]),
        ("zbe_decompress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t]),
        ("zbp_decompress", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int]),
        ("zbp_decompress_at", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int, C.c_int]),
        ("zbh_compress_params", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int, C.c_uint, C.POINTER(C.c_uint), C.c_int]),
        ("zbh_generate_sequences", C.c_size_t, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int, C.c_int]),
    ])
    if L is None:
        raise RuntimeError(f"{HOSTSIM_PATH} missing: run __graft_entry__.build()")
    return L


def _call_c(fn, data: bytes, level=None):
    cap = len(data) + (len(data) >> 8) + 1024
    out = C.create_string_buffer(cap)
    n = fn(out, cap, data, len(data), level) if level is not None else fn(out, cap, data, len(data))
    return out.raw[:n] if n <= ERR_MAX else -((1 << 64) - n)


def _call_d(fn, frame: bytes, cap: int):
    out = C.create_string_buffer(max(cap, 1))
    n = fn(out, cap, frame, len(frame))
    return out.raw[:n] if n <= ERR_MAX else -((1 << 64) - n)


def oracle_compress(data: bytes, level: int = 3):
    """Frame (bytes) or negative error code, from the plain-C restatement."""
    return _call_c(zso().zso_compress, data, level)


def _call_flags(fn, data: bytes, level: int, flags: int):
    cap = len(data) + (len(data) >> 8) + 1024
    out = C.create_string_buffer(cap)
    n = fn(out, cap, data, len(data), level, flags)
    return out.raw[:n] if n <= ERR_MAX else -((1 << 64) - n)


def oracle_compress_flags(data: bytes, level: int, checksum: bool = False, content_size: bool = True):
    return _call_flags(zso().zso_compress_flags, data, level, (1 if checksum else 0) | (0 if content_size else 2))


def hostsim_compress_flags(data: bytes, level: int, checksum: bool = False, content_size: bool = True, magicless: bool = False):
    return _call_flags(hostsim().zbh_compress_flags, data, level, (1 if checksum else 0) | (0 if content_size else 2) | (4 if magicless else 0))


def hostsim_decompress_magicless(frame: bytes, cap: int):
    out = C.create_string_buffer(max(cap, 1))
    n = hostsim().zbh_decompress_format(out, cap, frame, len(frame), 1)
    return out.raw[:n] if n <= ERR_MAX else -((1 << 64) - n)


@_recorded
def ref_decompress_magicless(frame: bytes, cap: int):
    """ZSTD_d_format = ZSTD_f_zstd1_magicless (J/ZstdDecompressCtx.setMagicless, N/jni_zstd.c:413-414)."""
    R = ref()
    dctx = R.ZSTD_createDCtx()
    try:
        assert R.ZSTD_DCtx_setParameter(dctx, 1000, 1) <= ERR_MAX
        out = C.create_string_buffer(max(cap, 1))
        n = R.ZSTD_decompressDCtx(dctx, out, cap, frame, len(frame))
        return out.raw[:n] if n <= ERR_MAX else -((1 << 64) - n)
    finally:
        R.ZSTD_freeDCtx(dctx)


@_recorded
def ref_compress_flags(data: bytes, level: int, checksum: bool = False, content_size: bool = True, magicless: bool = False):
    """The compiled reference through ZSTD_CCtx_setParameter + ZSTD_compress2 (what J/ZstdCompressCtx drives)."""
    R = ref()
    cctx = R.ZSTD_createCCtx()
    try:
        R.ZSTD_CCtx_setParameter(cctx, 100, level)
        if magicless:
            assert R.ZSTD_CCtx_setParameter(cctx, 10, 1) <= ERR_MAX      # ZSTD_c_format = ZSTD_f_zstd1_magicless
        R.ZSTD_CCtx_setParameter(cctx, 201, 1 if checksum else 0)
        R.ZSTD_CCtx_setParameter(cctx, 200, 1 if content_size else 0)
        cap = len(data) + (len(data) >> 8) + 1024
        out = C.create_string_buffer(cap)
        n = R.ZSTD_compress2(cctx, out, cap, data, len(data))
        return out.raw[:n] if n <= ERR_MAX else -((1 << 64) - n)
    finally:
        R.ZSTD_freeCCtx(cctx)


def oracle_decompress(frame: bytes, cap: int):
    return _call_d(zso().zso_decompress, frame, cap)


@_recorded
def ref_compress(data: bytes, level: int = 3):
    return _call_c(ref().ZSTD_compress, data, level)


@_recorded
def ref_decompress(frame: bytes, cap: int):
    return _call_d(ref().ZSTD_decompress, frame, cap)


def frame_header_prefixes(get_header, blob: bytes, fmt: int, lengths):
    """get_header (a ZSTD_getFrameHeader_advanced) on blob[:n] for every n of lengths: [result, header fields or None] per prefix."""
    from zstd_jni_b200._native import FrameHeader
    out = []
    for n in lengths:
        h = FrameHeader()
        r = get_header(C.byref(h), blob[:n], n, fmt)
        out.append([r, [h.frameContentSize, h.windowSize, h.blockSizeMax, h.frameType, h.headerSize, h.dictID, h.checksumFlag] if r == 0 else None])
    return out


@_recorded
def ref_frame_header_prefixes(blob: bytes, fmt: int, lengths: list):
    R = ref()
    R.ZSTD_getFrameHeader_advanced.restype = C.c_size_t
    R.ZSTD_getFrameHeader_advanced.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, C.c_int]
    return frame_header_prefixes(R.ZSTD_getFrameHeader_advanced, blob, fmt, lengths)


def hostsim_compress(data: bytes, level: int = 3):
    return _call_c(hostsim().zbh_compress, data, level)


def hostsim_decompress(frame: bytes, cap: int):
    return _call_d(hostsim().zbh_decompress, frame, cap)


def emu_compress(data: bytes, level: int = 3):
    """Kernel source on the emulated 32-lane warp (tests/hostsim/simt_emu.h)."""
    return _call_c(hostsim().zbe_compress, data, level)


def emu_decompress(frame: bytes, cap: int):
    return _call_d(hostsim().zbe_decompress, frame, cap)


def staged_decompress(frame: bytes, cap: int, emu: bool = False, misalign: int = 0):
    """The staged batch decoder (zb_decode_fast.cuh) on the host (1 lane) or on the 32-lane emulator; `misalign` = distance of the
    destination from a 16-byte boundary (a batch packs its outputs back to back)."""
    out = C.create_string_buffer(max(cap, 1))
    n = hostsim().zbp_decompress_at(out, cap, frame, len(frame), 1 if emu else 0, misalign)
    return out.raw[:n] if n <= ERR_MAX else -((1 << 64) - n)


def ref_stream_compress(data: bytes, level: int, slice_size: int = 131072, checksum: bool = False) -> bytes:
    """The reference's streaming path (what ZstdOutputStream drives): ZSTD_compressStream2 fed `slice_size`
    pieces then ZSTD_e_end; produces one multi-block frame with unknown content size."""
    R = ref()

    class Buf(C.Structure):
        _fields_ = [("p", C.c_void_p), ("size", C.c_size_t), ("pos", C.c_size_t)]

    cctx = R.ZSTD_createCCtx()
    R.ZSTD_CCtx_setParameter(cctx, 100, level)
    if checksum:
        R.ZSTD_CCtx_setParameter(cctx, 201, 1)
    out = bytearray()
    dst = C.create_string_buffer(1 << 18)
    pos = 0
    while True:
        piece = data[pos:pos + slice_size]
        pos += len(piece)
        last = pos >= len(data)
        src = C.create_string_buffer(piece, max(len(piece), 1))
        ib = Buf(C.cast(src, C.c_void_p), len(piece), 0)
        while True:
            ob = Buf(C.cast(dst, C.c_void_p), len(dst), 0)
            r = R.ZSTD_compressStream2(cctx, C.byref(ob), C.byref(ib), 2 if last else 0)
            assert r <= ERR_MAX, r
            out += dst.raw[:ob.pos]
            if (last and r == 0) or (not last and ib.pos == ib.size):
                break
        if last:
            break
    R.ZSTD_freeCCtx(cctx)
    return bytes(out)


# ---- sequences (ZSTD_Sequence records: offset, litLength, matchLength, rep -- 4 x u32)
@_recorded
def ref_generate_sequences(data: bytes, level: int):
    """ZSTD_generateSequences of the compiled reference: (n, 4) uint32 array, or a negative error code."""
    import numpy as np
    R = ref()
    cctx = R.ZSTD_createCCtx()
    try:
        R.ZSTD_CCtx_setParameter(cctx, 100, level)
        cap = R.ZSTD_sequenceBound(len(data)) + 2
        out = np.zeros((cap, 4), dtype=np.uint32)
        n = R.ZSTD_generateSequences(cctx, out.ctypes.data, cap, data, len(data))
        return out[:n].copy() if n <= ERR_MAX else -((1 << 64) - n)
    finally:
        R.ZSTD_freeCCtx(cctx)


def hostsim_generate_sequences(data: bytes, level: int, emu: bool = False):
    import numpy as np
    cap = len(data) // 3 + 16
    out = np.zeros((cap, 4), dtype=np.uint32)
    n = hostsim().zbh_generate_sequences(out.ctypes.data, cap, data, len(data), level, 1 if emu else 0)
    return out[:n].copy() if n <= ERR_MAX else -((1 << 64) - n)


# ---- explicit compression parameters (J/ZstdCompressCtx.setWindowLog ... setStrategy -> ZSTD_c_windowLog ... ZSTD_c_strategy)
CPARAM_IDS = {"windowLog": 101, "hashLog": 102, "chainLog": 103, "searchLog": 104, "minMatch": 105, "targetLength": 106, "strategy": 107}
CPARAM_ORDER = ("windowLog", "chainLog", "hashLog", "searchLog", "minMatch", "targetLength", "strategy")      # zb::CParams member order


@_recorded
def ref_compress_params(data: bytes, level: int, params: dict, checksum: bool = False):
    """The compiled reference: ZSTD_CCtx_setParameter for every explicit parameter, then ZSTD_compress2."""
    R = ref()
    cctx = R.ZSTD_createCCtx()
    try:
        R.ZSTD_CCtx_setParameter(cctx, 100, level)
        if checksum:
            R.ZSTD_CCtx_setParameter(cctx, 201, 1)
        for k, v in params.items():
            r = R.ZSTD_CCtx_setParameter(cctx, CPARAM_IDS[k], v)
            if r > ERR_MAX:
                return -((1 << 64) - r)
        cap = len(data) + (len(data) >> 8) + 1024
        out = C.create_string_buffer(cap)
        n = R.ZSTD_compress2(cctx, out, cap, data, len(data))
        return out.raw[:n] if n <= ERR_MAX else -((1 << 64) - n)
    finally:
        R.ZSTD_freeCCtx(cctx)


def hostsim_compress_params(data: bytes, level: int, params: dict, checksum: bool = False, emu: bool = False):
    ov = (C.c_uint * 7)(*[int(params.get(k, 0)) for k in CPARAM_ORDER])
    cap = len(data) + (len(data) >> 8) + 1024
    out = C.create_string_buffer(cap)
    n = hostsim().zbh_compress_params(out, cap, data, len(data), level, 1 if checksum else 0, ov, 1 if emu else 0)
    return out.raw[:n] if n <= ERR_MAX else -((1 << 64) - n)

"""Frame-format parameters of the JNI surface that only affect framing (SURVEY.md section 8f.3):
ZSTD_c_format / ZSTD_d_format = ZSTD_f_zstd1_magicless (J/ZstdCompressCtx.setMagicless, J/ZstdDecompressCtx.setMagicless,
N/jni_zstd.c:362-363,413-414), ZSTD_d_windowLogMax (J/ZstdInputStreamNoFinalizer.setLongMax, N/jni_zstd.c:403), the frame
header getters (N/jni_zstd.c:32-40,139) and ZSTD_getFrameProgression (N/jni_fast_zstd.c:373).

CPU: kernel source on the host against tests/golden/magicless.json (made by the compiled reference) and the oracle; the
host-side header parser against the reference on every prefix length.  GPU (-m gpu): the same through the C ABI.
"""
import ctypes as C
import hashlib
import io
import json
from pathlib import Path

import pytest

from tests.golden.make_golden import regenerate_input
from tests.oracle_util import (ERR_MAX, hostsim_compress_flags, hostsim_decompress_magicless, oracle_compress_flags, ref_compress_flags,
                               ref_decompress_magicless, same)

GOLDEN_DIR = Path(__file__).parent / "golden"
MAGICLESS = json.loads((GOLDEN_DIR / "magicless.json").read_text())


def _probe_blobs():
    data = regenerate_input({"kind": "corpus", "index": 1, "size": 20000})
    z = oracle_compress_flags(data, 3)[4:]
    full = oracle_compress_flags(data, 3)
    return data, {"truncated": z[:-1], "trailing": z + b"\x00", "tiny": z[:3], "reserved-bit": bytes([z[0] | 8]) + z[1:], "dst-too-small": z,
                  "with-magic": full, "two-frames": z + z}


def test_hostsim_magicless_frames_match_golden():
    for e in MAGICLESS["frames"]:
        data = regenerate_input(e["input"])
        z = hostsim_compress_flags(data, e["level"], e["checksum"], e["content_size"], magicless=True)
        assert not isinstance(z, int) and len(z) == e["size"] and hashlib.sha256(z).hexdigest() == e["sha256"], e
        assert z == oracle_compress_flags(data, e["level"], e["checksum"], e["content_size"])[4:]
        assert hostsim_decompress_magicless(z, len(data)) == data


def test_hostsim_magicless_decoder_error_codes_match_golden():
    data, blobs = _probe_blobs()
    for e in MAGICLESS["errors"]:
        r = hostsim_decompress_magicless(blobs[e["name"]], e["cap"])
        assert (r if isinstance(r, int) else len(r)) == e["result"], e["name"]
    assert hostsim_decompress_magicless(blobs["two-frames"], 40000) == data + data


def test_magicless_pins_against_reference():
    data, blobs = _probe_blobs()
    for name, blob in blobs.items():
        cap = 19999 if name == "dst-too-small" else 40000 if name == "two-frames" else 20000
        assert hostsim_decompress_magicless(blob, cap) == ref_decompress_magicless(blob, cap), name
    for n in (0, 1, 7, 255, 256, 65792, 131072):
        d = regenerate_input({"kind": "corpus", "index": 3, "size": n})
        for ck, cs in ((False, True), (True, False)):
            assert hostsim_compress_flags(d, 3, ck, cs, magicless=True) == ref_compress_flags(d, 3, ck, cs, True)


def test_frames_naming_a_dictionary_are_refused_like_the_reference():
    """A frame whose header carries a non-zero dictionary ID cannot be decoded without that dictionary: dictionary_wrong (32), from the fused
    decoder, the staged decoder (which hands such frames over) and the emulated warp; a dictID field of 0 is decoded normally."""
    from tests.oracle_util import emu_decompress, hostsim_decompress, staged_decompress
    data = regenerate_input({"kind": "corpus", "index": 1, "size": 20000})
    z = oracle_compress_flags(data, 3)
    named = z[:4] + bytes([z[4] | 1]) + b"\x07" + z[5:]
    zero_id = z[:4] + bytes([z[4] | 2]) + b"\x00\x00" + z[5:]
    for dec in (hostsim_decompress, emu_decompress, staged_decompress):
        assert dec(named, 20000) == -32 and dec(zero_id, 20000) == data
    from tests.oracle_util import ref_decompress
    assert ref_decompress(named, 20000) == -32 and ref_decompress(zero_id, 20000) == data


def test_frame_header_getters_host_side(reference_resources=None):
    """No GPU involved: ZSTD_getFrameHeader_advanced & co are host-side parsers of the C ABI."""
    from zstd_jni_b200 import _native as N
    from zstd_jni_b200.zstd import Zstd, ZstdException
    L = N.lib()
    data = regenerate_input({"kind": "corpus", "index": 1, "size": 70000})
    z = oracle_compress_flags(data, 3, checksum=True)
    h = Zstd.getFrameHeader(z)
    assert h == {"frameContentSize": 70000, "windowSize": 70000, "blockSizeMax": 70000, "frameType": 0, "headerSize": 9, "dictID": 0, "checksumFlag": 1}
    assert Zstd.getFrameHeader(z[4:], magicless=True) == {**h, "headerSize": 5}
    assert Zstd.getFrameContentSize(z[4:], magicless=True) == 70000 and Zstd.decompressedSize(z[4:], magicless=True) == 70000
    assert Zstd.getFrameContentSize(z, magicless=True) == 0            # N/jni_zstd.c:35-37: any header failure reads as 0
    nz = oracle_compress_flags(data, 3, content_size=False)
    h2 = Zstd.getFrameHeader(nz)
    assert h2["frameContentSize"] == (1 << 64) - 1 and h2["windowSize"] == 1 << 17 and h2["blockSizeMax"] == 1 << 17 and h2["headerSize"] == 6
    assert Zstd.getFrameContentSize(nz) == -1
    skip = b"\x53\x2a\x4d\x18" + (7).to_bytes(4, "little") + b"skipped"
    assert Zstd.getFrameHeader(skip) == {"frameContentSize": 7, "windowSize": 0, "blockSizeMax": 0, "frameType": 1, "headerSize": 8, "dictID": 3, "checksumFlag": 0}
    assert L.ZSTD_isSkippableFrame(skip, len(skip)) == 1 and L.ZSTD_isFrame(skip, len(skip)) == 1 and L.ZSTD_isFrame(z, len(z)) == 1 and L.ZSTD_isFrame(z[4:], 20) == 0
    with_dict = bytes.fromhex("28b52ffd") + bytes([0x23, 0x10]) + b"\x11\x22\x33\x44" + b"\x05" + b"\x01\x00\x00"
    assert Zstd.getDictIdFromFrame(with_dict) == 0x33221110 and Zstd.getDictIdFromFrame(z) == 0 and Zstd.getDictIdFromFrame(b"junk") == 0
    assert L.ZSTD_frameHeaderSize(with_dict, len(with_dict)) == 10 and N.error_code(L.ZSTD_frameHeaderSize(z, 4)) == 72
    with pytest.raises(ZstdException) as ei:
        Zstd.getFrameHeader(b"\x00" * 16)
    assert ei.value.getErrorCode() == 10
    with pytest.raises(ZstdException) as ei:
        Zstd.getFrameHeader(z[:4] + bytes([z[4] | 8]) + z[5:])
    assert ei.value.getErrorCode() == 14
    fh = N.FrameHeader()
    assert [L.ZSTD_getFrameHeader(C.byref(fh), z[:k], k) for k in (0, 3, 4, 5, 8, 9)] == [5, 5, 5, 9, 9, 0]
    assert [L.ZSTD_getFrameHeader_advanced(C.byref(fh), z[4:4 + k], k, 1) for k in (0, 1, 4, 5)] == [1, 5, 5, 0]
    assert N.error_code(L.ZSTD_getFrameHeader(C.byref(fh), b"\x28\xb5\x00", 3)) == 10


def test_frame_header_parser_matches_reference_on_every_prefix():
    from zstd_jni_b200 import _native as N
    from tests.oracle_util import frame_header_prefixes, ref_frame_header_prefixes
    L = N.lib()
    blobs = [f.read_bytes() for f in sorted(GOLDEN_DIR.glob("*.zst"))[::6]] + [(GOLDEN_DIR / "concat_skippable.zst").read_bytes()]
    d = regenerate_input({"kind": "corpus", "index": 1, "size": 131072})
    for n in (0, 5, 300, 70000, 131072):
        for ck, cs in ((False, True), (True, False)):
            z = oracle_compress_flags(d[:n], 3, ck, cs)[4:]
            assert z == ref_compress_flags(d[:n], 3, ck, cs, True)
            blobs.append(z)
    blobs.append(bytes.fromhex("28b52ffd") + bytes([0x23, 0x10]) + b"\x11\x22\x33\x44" + b"\x05" + b"\x01\x00\x00")
    blobs.append(bytes.fromhex("28b52ffd") + bytes([0x00, 0xFF]) + b"\x01\x00\x00")          # window too large
    for b in blobs:
        for fmt in (0, 1):
            lengths = [min(n, len(b)) for n in list(range(0, 20)) + [len(b)]]
            got = frame_header_prefixes(L.ZSTD_getFrameHeader_advanced, b, fmt, lengths)
            assert same(ref_frame_header_prefixes(b, fmt, lengths), got), (b[:12].hex(), fmt)


def test_dctx_parameter_bounds_host_side():
    from zstd_jni_b200 import _native as N
    L = N.lib()
    d = L.ZSTD_createDCtx()
    try:
        assert L.ZSTD_DCtx_setParameter(d, 100, 27) == 0 and L.ZSTD_DCtx_setParameter(d, 100, 0) == 0 and L.ZSTD_DCtx_setParameter(d, 1000, 1) == 0
        assert N.error_code(L.ZSTD_DCtx_setParameter(d, 100, 9)) == 42 and N.error_code(L.ZSTD_DCtx_setParameter(d, 100, 32)) == 42
        assert N.error_code(L.ZSTD_DCtx_setParameter(d, 1000, 2)) == 42
        assert N.error_code(L.ZSTD_DCtx_setParameter(d, 1001, 1)) == 40
    finally:
        L.ZSTD_freeDCtx(d)
    c = L.ZSTD_createCCtx()
    try:
        assert L.ZSTD_CCtx_setParameter(c, 10, 1) == 1 and N.error_code(L.ZSTD_CCtx_setParameter(c, 10, 2)) == 42
    finally:
        L.ZSTD_freeCCtx(c)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_gpu_magicless_contexts_match_golden():
    from zstd_jni_b200.zstd import Zstd, ZstdCompressCtx, ZstdDecompressCtx, ZstdException
    with ZstdCompressCtx() as c, ZstdDecompressCtx() as d:
        d.setMagicless(True)
        for e in MAGICLESS["frames"]:
            data = regenerate_input(e["input"])
            c.setLevel(e["level"]).setChecksum(e["checksum"]).setContentSize(e["content_size"]).setMagicless(True)
            z = c.compress(data)
            assert len(z) == e["size"] and hashlib.sha256(z).hexdigest() == e["sha256"], e
            assert d.decompress(z, len(data)) == data
            if e["content_size"]:
                assert Zstd.getFrameContentSize(z, magicless=True) == len(data)
            c.setMagicless(False)
            assert c.compress(data)[4:] == z
        data, blobs = _probe_blobs()
        for e in MAGICLESS["errors"]:
            dst = bytearray(e["cap"])
            r = d.decompressByteArray(dst, 0, e["cap"], blobs[e["name"]], 0, len(blobs[e["name"]]), raise_on_error=False)
            assert (r if r <= ERR_MAX else -((1 << 64) - r)) == e["result"], e["name"]
        d.setMagicless(False)                               # back to ZSTD_f_zstd1: a magicless frame is an unknown prefix
        with pytest.raises(ZstdException) as ei:
            d.decompress(blobs["dst-too-small"], 20000)
        assert ei.value.getErrorCode() == 10
        assert d.decompress(blobs["with-magic"], 20000) == data
        d.setMagicless(True)
        d.reset()                                           # ZSTD_reset_session_and_parameters restores the default format
        assert d.decompress(blobs["with-magic"], 20000) == data


@pytest.mark.gpu
def test_gpu_magicless_batch_option():
    from zstd_jni_b200 import corpus
    from zstd_jni_b200.zstd import ZstdBatchContext
    chunks = [corpus.chunk(i).tobytes() for i in range(12)] + [b"", b"abc", corpus.chunk(3)[:5000].tobytes()]
    with ZstdBatchContext(0) as ctx:
        ctx.setOption("magicless", 1)
        frames = ctx.compressBatch(chunks, 3)
        for c, f in zip(chunks, frames):
            assert f == oracle_compress_flags(c, 3)[4:]
        assert ctx.decompressBatch(frames, [len(c) for c in chunks]) == chunks
        two = ctx.decompressBatch([frames[0] + frames[1]], [len(chunks[0]) + len(chunks[1])])
        assert two == [chunks[0] + chunks[1]]
        stream, sizes = ctx.compressChunks(b"".join(chunks[:12]), 131072, 3)
        back, out_sizes = ctx.decompressFrames(stream, sizes, [131072] * 12)
        assert back.tobytes() == b"".join(chunks[:12])
        ctx.setOption("magicless", 0)
        assert ctx.compressBatch(chunks[:2], 3) == [oracle_compress_flags(c, 3) for c in chunks[:2]]
        assert ctx.decompressBatch(frames[:1], [131072], raise_on_error=False) == [-10]


class _Buf(C.Structure):
    _fields_ = [("p", C.c_void_p), ("size", C.c_size_t), ("pos", C.c_size_t)]


def _stream_decode(blob: bytes, window_log_max=None, magicless=False, out_cap=131072, feed=None):
    """ZSTD_decompressStream loop of J/ZstdInputStreamNoFinalizer.java:165-226 over the C ABI."""
    from zstd_jni_b200 import _native as N
    L = N.lib()
    d = L.ZSTD_createDStream()
    try:
        L.ZSTD_initDStream(d)
        if window_log_max is not None:
            assert L.ZSTD_DCtx_setParameter(d, 100, window_log_max) == 0
        if magicless:
            assert L.ZSTD_DCtx_setParameter(d, 1000, 1) == 0
        src = C.create_string_buffer(blob, max(len(blob), 1))
        dst = C.create_string_buffer(out_cap)
        out = bytearray()
        pos, feed = 0, feed or max(len(blob), 1)
        while True:
            ib = _Buf(C.cast(src, C.c_void_p).value + pos, min(feed, len(blob) - pos), 0)
            while True:
                ob = _Buf(C.cast(dst, C.c_void_p).value, out_cap, 0)
                r = L.ZSTD_decompressStream(d, C.byref(ob), C.byref(ib))
                if r > ERR_MAX:
                    return -((1 << 64) - r)
                out += dst.raw[: ob.pos]
                if ib.pos == ib.size and ob.pos < ob.size:
                    break
            pos += ib.size
            if pos >= len(blob):
                return bytes(out)
    finally:
        L.ZSTD_freeDStream(d)


@pytest.mark.gpu
def test_gpu_stream_window_log_max_and_magicless():
    """Outcomes pinned with the reference's ZSTD_decompressStream (window of stream_L3.zst: 2 MB, windowLog 21)."""
    man = json.loads((GOLDEN_DIR / "manifest.json").read_text())
    e = [x for x in man["decode_only"] if x["file"] == "stream_L3.zst"][0]
    blob = (GOLDEN_DIR / e["file"]).read_bytes()
    out = _stream_decode(blob)
    assert not isinstance(out, int) and hashlib.sha256(out).hexdigest() == e["sha256"]
    assert _stream_decode(blob, window_log_max=20) == -16 and _stream_decode(blob, window_log_max=10) == -16
    out = _stream_decode(blob, window_log_max=21, feed=50000)
    assert not isinstance(out, int) and hashlib.sha256(out).hexdigest() == e["sha256"]
    data = regenerate_input({"kind": "corpus", "index": 1, "size": 131072})
    z = oracle_compress_flags(data, 3)
    assert _stream_decode(z, window_log_max=16, out_cap=1000) == -16            # single segment: the window is the content
    assert _stream_decode(z, window_log_max=17, out_cap=1000) == data
    assert _stream_decode(z, window_log_max=10, out_cap=131072) == data          # fits the caller's buffer in one pass: no window needed
    assert _stream_decode(z[4:], magicless=True, out_cap=4096, feed=1000) == data
    assert _stream_decode(z[4:], out_cap=4096, feed=1000) == -10
    assert _stream_decode(z, magicless=True, out_cap=4096, feed=1000) == -14


@pytest.mark.gpu
def test_gpu_frame_progression_and_input_stream_long_max():
    from zstd_jni_b200 import _native as N
    from zstd_jni_b200.zstd import ZstdCompressCtx, ZstdInputStream, ZstdException
    L = N.lib()
    data = regenerate_input({"kind": "multi", "indices": [1, 9, 5], "size": 300000})
    with ZstdCompressCtx() as c:
        c.setLevel(3)
        assert c.getFrameProgression() == {"ingested": 0, "consumed": 0, "produced": 0, "flushed": 0, "currentJobID": 0, "nbActiveWorkers": 0}
        src = C.create_string_buffer(data, len(data))
        dst = C.create_string_buffer(1 << 19)
        ib = _Buf(C.cast(src, C.c_void_p).value, 200000, 0)
        ob = _Buf(C.cast(dst, C.c_void_p).value, 1000, 0)
        r = L.ZSTD_compressStream2(c._ptr, C.byref(ob), C.byref(ib), 0)
        assert r <= ERR_MAX
        p = c.getFrameProgression()
        assert p["ingested"] == ib.pos and p["consumed"] == 131072 * (ib.pos // 131072) and p["flushed"] == ob.pos == 1000 and p["produced"] > p["flushed"]
        ib.size = len(data)
        ob = _Buf(C.cast(dst, C.c_void_p).value + 1000, (1 << 19) - 1000, 0)
        while True:
            r = L.ZSTD_compressStream2(c._ptr, C.byref(ob), C.byref(ib), 2)
            assert r <= ERR_MAX
            if r == 0:
                break
        p = c.getFrameProgression()
        assert p["ingested"] == p["consumed"] == len(data) and p["produced"] == p["flushed"] == 1000 + ob.pos
        stream = dst.raw[: 1000 + ob.pos]
    with ZstdInputStream(io.BytesIO(stream)) as s:
        s.setLongMax(17)
        assert s.read() == data
    with ZstdInputStream(io.BytesIO((GOLDEN_DIR / "stream_L3.zst").read_bytes())) as s:
        s.setLongMax(12)
        with pytest.raises(ZstdException) as ei:
            s.read()
        assert ei.value.getErrorCode() == 16

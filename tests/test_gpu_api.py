"""The Python mirror of the Java API, on the GPU (-m gpu).  Modelled on the reference's own tests,
src/test/scala/Zstd.scala: round trips over sizes straddling a block (:20-111), dst-too-small errors
(:186-221), use-after-close (:1000-1020), Input/Output streams (:223-297, :426-488)."""
import io

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _inputs():
    rng = np.random.default_rng(3)
    from zstd_jni_b200 import corpus
    out = [b"", b"a", rng.integers(0, 256, 1000, dtype=np.uint8).tobytes(), corpus.chunk(0)[:70000].tobytes(), corpus.chunk(5).tobytes(),
           rng.integers(0, 256, 131072, dtype=np.uint8).tobytes(), corpus.chunk(2)[:130 * 1024].tobytes()]
    return out


@pytest.mark.parametrize("level", [1, 3])
def test_zstd_compress_decompress_roundtrip(level):        # Zstd.scala:26-36
    from zstd_jni_b200.zstd import Zstd
    from tests.oracle_util import oracle_compress
    for data in _inputs():
        z = Zstd.compress(data, level)
        assert z == oracle_compress(data, level)
        assert Zstd.getFrameContentSize(z) == len(data)
        assert Zstd.decompress(z, len(data)) == data


def test_manual_buffers_and_too_small_dst():                # Zstd.scala:38-53,186-221
    from zstd_jni_b200.zstd import Zstd, ZstdCompressCtx, ZstdDecompressCtx, ZstdException
    data = _inputs()[3]
    dst = bytearray(Zstd.compressBound(len(data)))
    n = Zstd.compressInto(dst, data, 3)
    assert not Zstd.isError(n)
    out = bytearray(len(data))
    assert Zstd.decompressInto(out, bytes(dst[:n])) == len(data) and bytes(out) == data
    small = bytearray(len(data) - 1)
    r = Zstd.decompressInto(small, bytes(dst[:n]))
    assert Zstd.isError(r) and Zstd.getErrorCode(r) == 70
    tiny = bytearray(10)
    r = Zstd.compressInto(tiny, data, 3)
    assert Zstd.isError(r) and Zstd.getErrorCode(r) == 70
    with ZstdDecompressCtx() as d, pytest.raises(ZstdException) as ei:
        d.decompress(bytes(dst[:n]), len(data) - 1)
    assert ei.value.getErrorCode() == 70
    with ZstdCompressCtx() as c:
        c.setLevel(3)
        buf = bytearray(200000)
        k = c.compressByteArray(buf, 100, 150000, b"junk" + data + b"junk", 4, len(data))     # offsets honoured (jni_fast_zstd.c:615-639)
        assert bytes(buf[100:100 + k]) == bytes(dst[:n])
        with pytest.raises(IndexError):
            c.compressByteArray(buf, 100, 10 ** 6, data, 0, len(data))


def test_checksum_and_content_size_flags():                 # J/ZstdCompressCtx.setChecksum / setContentSize (N/jni_fast_zstd.c:277-318)
    from zstd_jni_b200.zstd import Zstd, ZstdCompressCtx
    from tests.oracle_util import oracle_compress_flags
    for data in _inputs():
        for checksum, content_size in ((True, True), (False, False), (True, False)):
            with ZstdCompressCtx() as c:
                c.setLevel(3).setChecksum(checksum).setContentSize(content_size)
                z = c.compress(data)
            assert z == oracle_compress_flags(data, 3, checksum, content_size), (len(data), checksum, content_size)
            assert Zstd.decompress(z, len(data)) == data
            assert (Zstd.getFrameContentSize(z) == len(data)) == content_size or len(data) == 0
    bad = bytearray(z); bad[-1] ^= 0x40                      # corrupt the stored checksum of the last frame
    from zstd_jni_b200.zstd import ZstdException
    with pytest.raises(ZstdException) as ei:
        Zstd.decompress(bytes(bad), len(data))
    assert ei.value.getErrorCode() == 22                     # checksum_wrong


def test_multi_frame_extension_for_large_inputs():
    """> 128 KB is refused by default (no approximation of multi-block frames); ZSTDB200_c_multiFrame opts into one frame per 128 KB."""
    from zstd_jni_b200 import corpus
    from zstd_jni_b200.zstd import Zstd, ZstdCompressCtx
    from tests.oracle_util import oracle_compress, oracle_decompress
    data = b"".join(corpus.chunk(i).tobytes() for i in (0, 1, 5))[: 300000]
    with ZstdCompressCtx() as c:
        c.setLevel(3).setMultiFrame(True)
        z = c.compress(data)
    exp = b"".join(oracle_compress(data[o:o + 131072], 3) for o in range(0, len(data), 131072))
    assert z == exp                                          # every 128 KB piece is the reference's frame for that piece
    assert Zstd.decompress(z, len(data)) == data
    assert oracle_decompress(z, len(data)) == data           # any zstd decoder reads concatenated frames


def test_unsupported_parameters_are_reported():
    from zstd_jni_b200.zstd import ZstdCompressCtx, ZstdException
    data = _inputs()[3]
    with ZstdCompressCtx() as c:
        c.setLevel(19)
        with pytest.raises(ZstdException) as ei:
            c.compress(data)
        assert ei.value.getErrorCode() == 40
    with ZstdCompressCtx() as c:                             # > one block: outside the bit-exact scope => refused, not approximated
        with pytest.raises(ZstdException):
            c.compress(bytes(200000))


def test_use_after_close():                                  # Zstd.scala:1000-1020,1072-1080
    from zstd_jni_b200.zstd import ZstdCompressCtx, ZstdDecompressCtx
    c = ZstdCompressCtx(); c.close(); c.close()
    with pytest.raises(RuntimeError, match="Closed"):
        c.compress(b"abc")
    d = ZstdDecompressCtx(); d.close()
    with pytest.raises(RuntimeError, match="Closed"):
        d.decompress(b"abc", 3)


def test_output_and_input_streams():                         # Zstd.scala:223-297
    from zstd_jni_b200.zstd import ZstdInputStream, ZstdOutputStream
    from tests.oracle_util import oracle_decompress
    from zstd_jni_b200 import corpus
    data = b"".join(corpus.chunk(i).tobytes() for i in (0, 1, 2))[:300001]
    sink = io.BytesIO()
    with ZstdOutputStream(sink, 3) as zo:
        for k in range(0, len(data), 50000):
            zo.write(data[k:k + 50000])
        zo.flush()
    z = sink.getvalue()
    assert oracle_decompress(z, len(data)) == data           # any zstd decoder reads the independent-frames stream
    with ZstdInputStream(io.BytesIO(z)) as zi:
        got = b""
        while True:
            part = zi.read(70000)
            if not part:
                break
            got += part
    assert got == data
    # 1 byte at a time upstream (Zstd.scala:447-467)
    class OneByte(io.RawIOBase):
        def __init__(self, b): self.b = b; self.p = 0
        def read(self, n=-1):
            if self.p >= len(self.b): return b""
            self.p += 1; return self.b[self.p - 1:self.p]
    small = data[:40000]
    sink = io.BytesIO()
    with ZstdOutputStream(sink, 1) as zo:
        zo.write(small)
    with ZstdInputStream(OneByte(sink.getvalue())) as zi:
        assert zi.read() == small
    # empty stream
    sink = io.BytesIO()
    ZstdOutputStream(sink, 3).close()
    assert oracle_decompress(sink.getvalue(), 0) == b""


def _frames_of(z: bytes):
    from zstd_jni_b200.zstd import Zstd
    out = []; pos = 0
    while pos < len(z):
        n = Zstd.findFrameCompressedSize(z[pos:]); out.append(z[pos:pos + n]); pos += n
    return out


def test_streams_batch_whole_blocks_and_frames():
    """The stream layer hands every whole block / frame offered in one call to the batch kernels (one launch chain per call, not per
    block), keeps one frame per 128 KB block -- each byte-identical to the one-shot frame of that block --, writes no spurious empty
    frame after a stream that ends on a block boundary, and reads back through both stream decoders."""
    import numpy as np
    from zstd_jni_b200 import corpus
    from zstd_jni_b200.zstd import (ByteBuffer, ZstdBatchContext, ZstdDirectBufferCompressingStream, ZstdDirectBufferDecompressingStream,
                                     ZstdInputStream, ZstdOutputStream)
    from tests.oracle_util import oracle_compress, oracle_decompress
    data = b"".join(corpus.chunk(i).tobytes() for i in range(24)) + corpus.chunk(3)[:50001].tobytes()      # 24 blocks + a tail
    # ZstdOutputStream: one big write
    sink = io.BytesIO()
    with ZstdBatchContext(0) as probe:
        pass
    with ZstdOutputStream(sink, 3) as zo:
        zo.write(data)
    z = sink.getvalue()
    frames = _frames_of(z)
    assert len(frames) == 25
    for k, f in enumerate(frames):
        assert f == oracle_compress(data[k * 131072:(k + 1) * 131072], 3), k
    assert oracle_decompress(z, len(data)) == data
    # a stream that is a whole number of blocks has exactly that many frames (no empty trailer); an empty stream has one
    sink = io.BytesIO()
    with ZstdOutputStream(sink, 3) as zo:
        zo.write(data[:131072])
    assert len(_frames_of(sink.getvalue())) == 1
    sink = io.BytesIO()
    with ZstdOutputStream(sink, 1) as zo:
        zo.write(data[:131072]); zo.write(data[131072:2 * 131072])
    assert len(_frames_of(sink.getvalue())) == 2
    # direct buffers both ways: the whole source goes to every native call
    src = ByteBuffer.allocateDirect(len(data)); src.array[:] = np.frombuffer(data, dtype=np.uint8)
    tgt = ByteBuffer.allocateDirect(len(data) + 4096)
    with ZstdDirectBufferCompressingStream(tgt, 3) as zc:
        zc.compress(src)
    tgt.flip()
    z2 = tgt.array[: tgt.limit()].tobytes()
    assert z2 == z
    back = ByteBuffer.allocateDirect(len(data) + 1)
    zd = ZstdDirectBufferDecompressingStream(tgt)
    while zd.hasRemaining():
        if zd.read(back) == 0 and not back.hasRemaining():
            break
    zd.close()
    assert back.position() == len(data) and back.array[: len(data)].tobytes() == data
    # small target buffer: the pending output is handed out piecewise
    class Drain(ZstdDirectBufferCompressingStream):
        def __init__(self, t, lvl): super().__init__(t, lvl); self.got = []
        def flushBuffer(self, b): b.flip(); self.got.append(b.array[: b.limit()].tobytes()); b.clear(); return b
    small = ByteBuffer.allocateDirect(ZstdDirectBufferCompressingStream.recommendedOutputBufferSize())
    src.position(0)
    dr = Drain(small, 3); dr.compress(src); dr.close()
    assert b"".join(dr.got) == z
    # ZstdInputStream over the multi-frame stream, odd read sizes
    with ZstdInputStream(io.BytesIO(z)) as zi:
        got = b""
        while True:
            part = zi.read(333333)
            if not part:
                break
            got += part
    assert got == data
    # a cut stream is reported, not padded
    with ZstdInputStream(io.BytesIO(z[:-5])) as zi:
        with pytest.raises(IOError):
            while zi.read(1 << 20):
                pass


def test_async_begin_end_api_overlaps_slots():
    """zstdb200_*_begin / _end: two batches in flight on two work sets give the same bytes as the synchronous calls."""
    import ctypes as C
    import numpy as np
    from zstd_jni_b200 import corpus
    from zstd_jni_b200.zstd import ZstdBatchContext
    n = 48
    a = corpus.corpus(n).reshape(-1); b = np.ascontiguousarray(a[::-1][: 40 * 131072 + 777])
    with ZstdBatchContext(0) as ctx:
        sa, fa = ctx.compressChunks(a, 131072, 3)
        sb, fb = ctx.compressChunks(b, 131072, 3)
        outA = np.empty(a.size + 65536, dtype=np.uint8); outB = np.empty(b.size + 65536, dtype=np.uint8)
        szA = (C.c_size_t * n)(); szB = (C.c_size_t * 41)()
        ctx.compressChunksBegin(0, a, 131072, 3)
        ctx.compressChunksBegin(1, b, 131072, 3)
        ta = ctx.compressChunksEnd(0, outA, szA)
        ctx.compressChunksBegin(0, a, 131072, 1)          # slot 0 is free again while slot 1 is still out
        tb = ctx.compressChunksEnd(1, outB, szB)
        tc = ctx.compressChunksEnd(0, np.empty(a.size + 65536, dtype=np.uint8))
        assert outA[:ta].tobytes() == sa.tobytes() and list(szA) == [int(x) for x in fa]
        assert outB[:tb].tobytes() == sb.tobytes() and list(szB) == [int(x) for x in fb]
        assert tc > 0
        # decompression: both streams in flight
        backA = np.empty(a.size, dtype=np.uint8); backB = np.empty(b.size, dtype=np.uint8)
        capA = (C.c_size_t * n)(*([131072] * n)); capB = (C.c_size_t * 41)(*([131072] * 40 + [777]))
        resA = (C.c_size_t * n)(); resB = (C.c_size_t * 41)()
        ctx.decompressFramesBegin(2, sa, szA, backA, capA)
        ctx.decompressFramesBegin(3, sb, szB, backB, capB)
        ctx.decompressFramesEnd(3, resB); ctx.decompressFramesEnd(2, resA)
        assert (backA == a).all() and (backB == b).all() and list(resB)[-1] == 777
        with pytest.raises(Exception):
            ctx.compressChunksEnd(2, outA)                # nothing queued on that slot: stage_wrong


def test_overlapped_stages_and_kernel_fifo_keep_the_bytes():
    """The entropy stage beside the parse (programmatic dependent launch + completion queue) and the one-operation-in-the-kernels rule
    are scheduling choices: frames are the same bytes with either switched off, for batch sizes around the residency of the parse grid,
    several levels, and two work sets in flight."""
    import ctypes as C
    import numpy as np
    from zstd_jni_b200 import corpus
    from zstd_jni_b200.zstd import ZstdBatchContext
    with ZstdBatchContext(0) as ctx:
        def both(n, level, start):
            data = corpus.corpus(n, start=start).reshape(-1)
            out = []
            for overlap, fifo in ((1, 1), (0, 1), (1, 0)):
                ctx.setOption("entropy_overlap", overlap); ctx.setOption("kernel_fifo", fifo)
                s, f = ctx.compressChunks(data, 131072, level)
                out.append((s.tobytes(), [int(x) for x in f]))
            ctx.setOption("entropy_overlap", 1); ctx.setOption("kernel_fifo", 1)
            return out
        for n, level, start in ((1, 3, 0), (7, 3, 3), (300, 3, 16), (129, 1, 5), (65, 9, 9), (4800, 3, 0)):
            a, b, c = both(n, level, start)
            assert a == b == c, (n, level)
        # the same batch twice in a row on two work sets: results do not depend on what else is queued
        data = corpus.corpus(400, start=21).reshape(-1)
        want, fw = ctx.compressChunks(data, 131072, 3)
        o0 = np.empty(data.size + 65536, dtype=np.uint8); o1 = np.empty(data.size + 65536, dtype=np.uint8)
        ctx.compressChunksBegin(0, data, 131072, 3); ctx.compressChunksBegin(1, data, 131072, 3)
        t0 = ctx.compressChunksEnd(0, o0); t1 = ctx.compressChunksEnd(1, o1)
        assert o0[:t0].tobytes() == want.tobytes() == o1[:t1].tobytes()


def test_input_stream_reads_reference_golden():   # Zstd.scala:426-446
    from tests.golden.make_golden_xml import is_xml_sample, xml_frame
    from zstd_jni_b200.zstd import ZstdInputStream
    with ZstdInputStream(io.BytesIO(xml_frame("xml-3.zst"))) as zi:
        assert is_xml_sample(zi.read())

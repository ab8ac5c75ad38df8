"""Parity tests proper (-m gpu): the CUDA path, called through the C ABI, against the oracle on the same
inputs, against the committed golden fixtures, and -- at BASELINE.json's full sizes -- through
size-independent properties (round trip, frame-size bookkeeping, checksum of checksums)."""
import hashlib
import io
import json
from pathlib import Path

import numpy as np
import pytest

from tests import cases
from tests.golden.make_golden_xml import SAMPLE, is_xml_sample, xml_frame
from tests.oracle_util import oracle_compress, oracle_decompress, ref_compress

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).parent / "golden"


@pytest.fixture(scope="module")
def ctx():
    from zstd_jni_b200.zstd import ZstdBatchContext
    c = ZstdBatchContext(0)
    yield c
    c.close()


def _expected(data, level):
    r = oracle_compress(data, level)
    assert ref_compress(data, level) == r
    return r


@pytest.mark.parametrize("level", [3, 1, 4, 2, -1, 5, 7, 9, 12])
def test_compress_bit_exact_vs_oracle(ctx, level):
    todo = cases.special_cases() + cases.corpus_cases(32) + cases.edge_cases()
    if level >= 11:
        todo = [t for t in todo if len(t[1]) > 16384]
    frames = ctx.compressBatch([d for _, d in todo], level)
    assert ctx.kernelLaunches() > 0
    for (name, data), got in zip(todo, frames):
        assert got == _expected(data, level), (name, level)


def test_unsupported_levels_fail_loudly(ctx):
    from zstd_jni_b200.zstd import ZstdException
    with pytest.raises(ZstdException) as ei:
        ctx.compressBatch([b"x" * 1000], 11)         # <= 16 KB at level 11: btopt (optimal parser), not built
    assert ei.value.getErrorCode() == 40
    with pytest.raises(ZstdException) as ei:
        ctx.compressBatch([b"x" * 100000], 13)       # btopt
    assert ei.value.getErrorCode() == 40


def test_golden_fixtures(ctx):
    man = json.loads((GOLDEN / "manifest.json").read_text())
    from tests.golden.make_golden import regenerate_input
    by_level = {}
    for e in man["oneshot"]:
        by_level.setdefault(e["level"], []).append(e)
    for level, es in by_level.items():
        datas = [regenerate_input(e["input"]) for e in es]
        frames = ctx.compressBatch(datas, level)
        for e, d, f in zip(es, datas, frames):
            assert f == (GOLDEN / e["file"]).read_bytes(), e["file"]
        back = ctx.decompressBatch([(GOLDEN / e["file"]).read_bytes() for e in es], [len(d) for d in datas])
        assert back == datas
    blobs = [(GOLDEN / e["file"]).read_bytes() for e in man["decode_only"]]
    outs = ctx.decompressBatch(blobs, [e["size"] for e in man["decode_only"]])
    for e, o in zip(man["decode_only"], outs):
        assert hashlib.sha256(o).hexdigest() == e["sha256"], e["file"]
    errs = ctx.decompressBatch([(GOLDEN / e["file"]).read_bytes() for e in man["errors"]], [e["cap"] for e in man["errors"]], raise_on_error=False)
    for e, r in zip(man["errors"], errs):
        assert r == -e["code"], (e["file"], r)


def test_decoder_matches_oracle_on_corruptions(ctx):
    from zstd_jni_b200 import corpus
    rng = np.random.default_rng(5)
    blobs, caps, exp = [], [], []
    for idx in (0, 1, 2, 4, 5, 7):
        data = corpus.chunk(idx)[:50000].tobytes()
        z = oracle_compress(data, 3)
        for _ in range(48):
            zz = bytearray(z)
            k = int(rng.integers(0, len(zz))); zz[k] ^= 1 << int(rng.integers(0, 8))
            if rng.random() < 0.2:
                zz = zz[: int(rng.integers(1, len(zz)))]
            blobs.append(bytes(zz)); caps.append(len(data)); exp.append(oracle_decompress(bytes(zz), len(data)))
    got = ctx.decompressBatch(blobs, caps, raise_on_error=False)
    for k, (e, g) in enumerate(zip(exp, got)):
        assert e == g, (k, e if isinstance(e, int) else "ok", g if isinstance(g, int) else "ok")


def _literal_payload(z: bytes):
    """(first, end) byte range of the compressed-literals payload (Huffman tree description + streams) of a one-block frame, or None."""
    fhd = z[4]; single = (fhd >> 5) & 1; fcs = fhd >> 6; did = fhd & 3
    pos = 5 + (0 if single else 1) + (4 if did == 3 else did) + ((1 << fcs) if fcs else (1 if single else 0))
    bh = z[pos] | (z[pos + 1] << 8) | (z[pos + 2] << 16)
    if (bh >> 1) & 3 != 2:
        return None
    blk = pos + 3
    b0 = z[blk]; typ = b0 & 3; lhl = (b0 >> 2) & 3
    if typ < 2:
        return None
    lhc = int.from_bytes(z[blk:blk + 5], "little")
    if lhl < 2: lh, csz = 3, (lhc >> 14) & 0x3FF
    elif lhl == 2: lh, csz = 4, (lhc >> 18) & 0x3FFF
    else: lh, csz = 5, (lhc >> 22) & 0x3FFFF
    return blk + lh, blk + lh + csz


def test_decoder_matches_the_compiled_reference_on_corruptions(ctx):
    """The same single-bit corruptions judged by the reference itself (oracle/_ref), not by the restatement.  One class of input is
    allowed to differ, exactly as DESIGN.md section 5 documents it: a flipped bit INSIDE the compressed-literals payload, where this
    decoder demands that every Huffman stream ends on its first bit (corruption_detected) while the reference's fast 4-stream loop
    (N/decompress/huf_decompress.c:219,236,281-300,840-893) may hand back bytes or a later error.  Anything else must agree."""
    from zstd_jni_b200 import corpus
    from tests.oracle_util import ref_decompress
    rng = np.random.default_rng(11)
    blobs, caps, exp, where, hdr = [], [], [], [], []
    for idx in (0, 1, 2, 3, 4, 5, 7, 9):
        data = corpus.chunk(idx)[:60000].tobytes()
        for level in (3, 1):
            z = oracle_compress(data, level)
            assert z == ref_compress(data, level), (idx, level)
            lit = _literal_payload(z)
            for _ in range(40):
                zz = bytearray(z)
                k = int(rng.integers(0, len(zz))); zz[k] ^= 1 << int(rng.integers(0, 8))
                blobs.append(bytes(zz)); caps.append(len(data)); exp.append(ref_decompress(bytes(zz), len(data)))
                where.append(lit is not None and lit[0] <= k < lit[1]); hdr.append(4 <= k < 9)
    got = ctx.decompressBatch(blobs, caps, raise_on_error=False)
    allowed = header = 0
    for k, (e, g) in enumerate(zip(exp, got)):
        if e == g:
            continue
        if hdr[k] and isinstance(e, int) and isinstance(g, int) and {e, g} <= {-20, -70}:
            header += 1          # second documented class: a damaged content-size / window field; the reference trips over its literal-buffer
            continue             # placement inside dst (dstSize_tooSmall), this decoder over the size check (corruption_detected) or vice versa
        assert where[k] and g == -20, (k, e if isinstance(e, int) else "bytes", g if isinstance(g, int) else "bytes")
        allowed += 1
    assert allowed <= len(blobs) // 4 and header <= len(blobs) // 50, (allowed, header)        # minorities (~8 % and < 1 % of random flips)


def test_decodes_reference_streams(ctx):
    """The reference's streaming path over the 256 KB sample of `xml` (tests/golden/xml), with and without checksums."""
    blobs = [xml_frame(f"xml-{lv}{'-xxh' if cs else ''}.zst") for lv in (1, 3, 9, 15) for cs in (False, True)]
    outs = ctx.decompressBatch(blobs, [SAMPLE] * len(blobs))
    assert all(is_xml_sample(o) for o in outs)


def test_reference_golden_resources(ctx):
    names = ["xml-1.zst", "xml-3.zst", "xml-6.zst", "xml-9.zst", "xml-1-sized.zst"]
    outs = ctx.decompressBatch([xml_frame(n) for n in names], [SAMPLE] * len(names))
    assert all(is_xml_sample(o) for o in outs)


def test_full_size_config_properties(ctx):
    """configs[1] shape at a CI-sized scale (2048 x 128 KB = 256 MiB): frames == oracle on a sample,
    sizes consistent, exact round trip, digest of digests stable across two runs."""
    from zstd_jni_b200 import corpus
    n = 2048
    data = corpus.corpus(n)
    stream, sizes = ctx.compressChunks(data.reshape(-1), 131072, 3)
    assert int(sizes.sum()) == stream.size and len(sizes) == n
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    for i in list(range(0, 64)) + list(range(64, n, 37)):
        assert stream[offs[i]:offs[i + 1]].tobytes() == oracle_compress(data[i].tobytes(), 3), i
    out, osz = ctx.decompressFrames(stream, sizes, [131072] * n)
    assert (osz == 131072).all() and np.array_equal(out.reshape(n, -1), data)
    stream2, sizes2 = ctx.compressChunks(data.reshape(-1), 131072, 3)
    assert hashlib.sha256(stream.tobytes()).digest() == hashlib.sha256(stream2.tobytes()).digest() and np.array_equal(sizes, sizes2)
    # the packed stream is one legal multi-frame zstd stream: the CPU oracle reads a prefix of it whole
    k = 16
    assert oracle_decompress(stream[: offs[k]].tobytes(), k * 131072) == data[:k].tobytes()


def test_mixed_level_frame_batches(ctx):
    """configs[3] shape at a CI-sized scale: pre-built frames of mixed entropy (levels cycling 1 / 3 / 9, ragged sizes, a sample checked
    against the oracle), decoded in batches of several sizes; every batch must regenerate exactly its chunks."""
    from zstd_jni_b200 import corpus
    rng = np.random.default_rng(21)
    n = 600
    chunks = [corpus.chunk(j)[: (131072 if j % 5 else int(rng.integers(1, 131072)))].tobytes() for j in range(n)]
    frames = [None] * n
    for k, level in enumerate((1, 3, 9)):
        idx = list(range(k, n, 3))
        for j, f in zip(idx, ctx.compressBatch([chunks[j] for j in idx], level)):
            frames[j] = f
        for j in idx[:6]:
            assert frames[j] == oracle_compress(chunks[j], level), (j, level)
    order = rng.permutation(n)
    for batch in (64, 512, n):
        for lo in range(0, n, batch):
            sel = order[lo:lo + batch]
            stream = np.frombuffer(b"".join(frames[j] for j in sel), dtype=np.uint8)
            out, osz = ctx.decompressFrames(stream, [len(frames[j]) for j in sel], [len(chunks[j]) for j in sel])
            assert [int(x) for x in osz] == [len(chunks[j]) for j in sel]
            assert out.tobytes() == b"".join(chunks[j] for j in sel), (batch, lo)


def test_staged_and_fused_decoders_agree(ctx):
    """The staged batch decoder (default) and the fused kernel must return the same bytes and the same
    error codes on a mixed bag: valid single-block frames, multi-block streams, corrupted frames."""
    from zstd_jni_b200 import corpus
    rng = np.random.default_rng(9)
    blobs, caps = [], []
    for i in range(48):
        data = corpus.chunk(i)[: int(rng.integers(1, 131073))].tobytes()
        z = oracle_compress(data, 3 if i % 3 else 1)
        blobs.append(z); caps.append(len(data))
        zz = bytearray(z); k = int(rng.integers(0, len(zz))); zz[k] ^= 1 << int(rng.integers(0, 8))
        blobs.append(bytes(zz)); caps.append(len(data))
        blobs.append(z); caps.append(max(0, len(data) - 3))
    blobs.append(blobs[0] + blobs[3]); caps.append(caps[0] + caps[3])          # two frames in one item -> fused path
    ctx.setOption("dec_pipeline", 1)
    a = ctx.decompressBatch(blobs, caps, raise_on_error=False)
    ctx.setOption("dec_pipeline", 0)
    b = ctx.decompressBatch(blobs, caps, raise_on_error=False)
    ctx.setOption("dec_pipeline", 1)
    exp = [oracle_decompress(z, c) for z, c in zip(blobs, caps)]
    assert a == exp and b == exp


def test_device_resident_api(ctx):
    import torch
    from zstd_jni_b200 import _native, corpus
    L = _native.lib()
    n = 300
    data = corpus.corpus(n, size=100000)
    dev = torch.device("cuda:0")
    d_src = torch.from_numpy(data.reshape(-1)).to(dev)
    d_off = torch.arange(0, (n + 1) * 100000, 100000, dtype=torch.int64, device=dev)
    stride = (L.ZSTD_compressBound(100000) + 32 + 63) // 64 * 64
    d_slots = torch.empty(n * stride, dtype=torch.uint8, device=dev)
    d_sizes = torch.zeros(n, dtype=torch.int64, device=dev)
    d_out = torch.empty(n * stride, dtype=torch.uint8, device=dev)
    d_ooff = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    d_back = torch.zeros(n * 100000, dtype=torch.uint8, device=dev)
    d_res = torch.zeros(n, dtype=torch.int64, device=dev)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        assert L.zstdb200_compress_device(ctx.handle, 3, n, d_src.data_ptr(), d_off.data_ptr(), d_slots.data_ptr(), stride, d_sizes.data_ptr(), s.cuda_stream) == 0
        assert L.zstdb200_compact_device(ctx.handle, n, d_slots.data_ptr(), stride, d_sizes.data_ptr(), d_out.data_ptr(), d_ooff.data_ptr(), s.cuda_stream) == 0
        assert L.zstdb200_decompress_device(ctx.handle, n, d_out.data_ptr(), d_ooff.data_ptr(), d_back.data_ptr(), d_off.data_ptr(), d_res.data_ptr(), s.cuda_stream) == 0
    s.synchronize()
    assert torch.equal(d_back, d_src) and bool((d_res == 100000).all())
    sizes = d_sizes.cpu().numpy(); ooff = d_ooff.cpu().numpy(); packed = d_out.cpu().numpy()
    assert (np.diff(ooff) == sizes).all()
    for i in (0, 1, 7, 150, 299):
        assert packed[ooff[i]:ooff[i + 1]].tobytes() == oracle_compress(data[i].tobytes(), 3)

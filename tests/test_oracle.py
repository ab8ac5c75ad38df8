"""CPU tests of the oracle (plain-C restatement): pinned against the reference's own golden vectors,
against the reference compiled in place (oracle/_ref) and against the committed fixtures in tests/golden."""
import hashlib
import json
from pathlib import Path

import pytest

from tests import cases
from tests.golden.make_golden_xml import LEVELS, SAMPLE, is_xml_sample, xml_frame
from tests.oracle_util import oracle_compress, oracle_decompress, ref, ref_compress, ref_decompress, zso

GOLDEN = Path(__file__).parent / "golden"


def test_reference_golden_decode():
    """T/scala/Zstd.scala:426-676 : xml-{1,3,6,9}.zst (+ sized / x2 / combined variants) must regenerate `xml` (tests/golden/xml: the
    reference's vectors remade on a 256 KB sample of `xml`)."""
    for name in ["xml-1.zst", "xml-3.zst", "xml-6.zst", "xml-9.zst", "xml-1-sized.zst", "xml-advanced.zst"]:
        assert is_xml_sample(oracle_decompress(xml_frame(name), SAMPLE)), name
    for name in ["xml-1.zst", "xml-1-sized.zst"]:                  # xml-1x2.zst, xml-1-sizedx2.zst
        assert is_xml_sample(oracle_decompress(xml_frame(name) * 2, 2 * SAMPLE), copies=2), name
    small = xml_frame("xmlsmall")
    assert oracle_decompress(xml_frame("xmlsmall-sized.zst"), len(small)) == small


def test_committed_golden_vectors():
    """tests/golden/manifest.json was produced by tests/golden/make_golden.py from the compiled reference."""
    man = json.loads((GOLDEN / "manifest.json").read_text())
    from tests.golden.make_golden import regenerate_input
    for e in man["oneshot"]:
        data = regenerate_input(e["input"])
        assert hashlib.sha256(data).hexdigest() == e["input_sha256"]
        frame = (GOLDEN / e["file"]).read_bytes()
        assert oracle_compress(data, e["level"]) == frame, e["file"]
        assert oracle_decompress(frame, len(data)) == data, e["file"]
    for e in man["decode_only"]:
        frame = (GOLDEN / e["file"]).read_bytes()
        out = oracle_decompress(frame, e["size"])
        assert not isinstance(out, int), (e["file"], out)
        assert hashlib.sha256(out).hexdigest() == e["sha256"], e["file"]
    for e in man["errors"]:
        frame = (GOLDEN / e["file"]).read_bytes()
        assert oracle_decompress(frame, e["cap"]) == -e["code"], e["file"]


@pytest.mark.parametrize("level", [1, 2, 3, 4, -1, -5, 5, 6, 7, 9, 10, 12])
def test_oracle_matches_compiled_reference(level):
    if ref() is not None:
        assert ref().ZSTD_versionString() == b"1.5.7"
    todo = cases.special_cases() + cases.corpus_cases(16) + cases.edge_cases(classes=(0, 4))
    for name, data in todo:
        if level >= 11 and len(data) <= 16384:
            assert oracle_compress(data, level) == -40     # <=16 KB table, level 11+: optimal parser (btopt), not restated
            continue
        got = oracle_compress(data, level)
        assert got == ref_compress(data, level), (name, level)
        assert oracle_decompress(got, len(data)) == data, (name, level)


@pytest.mark.parametrize("checksum,content_size", [(True, True), (False, False), (True, False)])
def test_oracle_frame_flags_match_reference(checksum, content_size):
    """ZSTD_c_checksumFlag / ZSTD_c_contentSizeFlag as J/ZstdCompressCtx.setChecksum / setContentSize set them."""
    from tests.oracle_util import oracle_compress_flags, ref_compress_flags
    for name, data in cases.special_cases()[:4] + cases.corpus_cases(6) + cases.edge_cases(classes=(0, 4), sizes=[0, 1, 7, 255, 256, 1000, 65791, 65792, 131072]):
        for level in (3, 1, 9):
            if level == 9 and 0 < len(data) <= 16384 and False:
                continue
            got = oracle_compress_flags(data, level, checksum, content_size)
            assert got == ref_compress_flags(data, level, checksum, content_size), (name, level)
            assert oracle_decompress(got, len(data)) == data


def test_oracle_decodes_reference_streams():
    """multi-block frames with cross-block matches, repeat modes, checksums (what ZstdOutputStream emits): the reference's streaming
    path over the 256 KB sample of `xml` (tests/golden/xml)."""
    for level in LEVELS:
        for name in (f"xml-{level}.zst", f"xml-{level}-xxh.zst"):
            assert is_xml_sample(oracle_decompress(xml_frame(name), SAMPLE)), name
    z = xml_frame("xml-3.zst")
    assert is_xml_sample(oracle_decompress(z + z, 2 * SAMPLE), copies=2)          # two frames
    skippable = b"\x50\x2a\x4d\x18" + (5).to_bytes(4, "little") + b"hello"
    assert is_xml_sample(oracle_decompress(skippable + z + skippable, SAMPLE))


def test_oracle_error_codes_match_reference():
    from zstd_jni_b200 import corpus
    data = corpus.chunk(0).tobytes()
    z = oracle_compress(data, 3)
    assert z == ref_compress(data, 3)
    probes = [z[:-1], z[:100], z[:5], z[:3], b"", b"\x00" * 20, z[:9] + b"\xff" + z[10:], z + b"\x01", z[:40] + bytes(64) + z[104:]]
    for k, p in enumerate(probes):
        a = ref_decompress(p, len(data)); b = oracle_decompress(p, len(data))
        assert (a == b) or (isinstance(a, int) and isinstance(b, int)), (k, a if isinstance(a, int) else "bytes", b if isinstance(b, int) else len(b))
    assert ref_decompress(z, len(data) - 1) == oracle_decompress(z, len(data) - 1) == -70   # dstSize_tooSmall
    assert oracle_decompress(z[:-1], len(data)) == ref_decompress(z[:-1], len(data))


def test_oracle_bounds_and_frame_queries():
    L = zso()
    for n in (0, 1, 1000, 131071, 131072, 1 << 20):
        assert L.zso_compressBound(n) == n + (n >> 8) + (((128 << 10) - n) >> 11 if n < (128 << 10) else 0)
    from zstd_jni_b200 import corpus
    data = corpus.chunk(2)[:50000].tobytes()
    z = oracle_compress(data, 3)
    assert L.zso_findFrameCompressedSize(z + b"junk", len(z) + 4) == len(z)
    assert L.zso_getFrameContentSize(z, len(z)) == len(data)

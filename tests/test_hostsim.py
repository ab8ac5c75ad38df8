"""CPU tests of the *kernel source itself*: zstd_jni_b200/csrc/*.cuh instantiated with a 1-lane warp
context (tests/hostsim/zb_hostsim.cpp) must agree with the oracle byte for byte.  This is how format
logic is iterated on without a GPU; the CUDA build of the same source is checked by the -m gpu tests."""
import hashlib
import json
from pathlib import Path

import pytest

from tests import cases
from tests.golden.make_golden_xml import SAMPLE, is_xml_sample, xml_frame
from tests.oracle_util import emu_compress, emu_decompress, hostsim_compress, hostsim_decompress, oracle_compress, oracle_decompress

GOLDEN = Path(__file__).parent / "golden"


@pytest.mark.parametrize("level", [3, 1, 4, 2, -1, -7, 5, 6, 9, 12])
def test_hostsim_encoder_matches_oracle(level):
    todo = cases.special_cases() + cases.corpus_cases(16) + cases.edge_cases(classes=(0, 2, 4, 5, 7))
    if level >= 5:       # lazy levels (row match finder): keep the CPU suite short, the big inputs are what they are for
        todo = cases.special_cases() + cases.corpus_cases(8) + cases.edge_cases(classes=(0, 4), sizes=[7, 100, 1024, 5000, 16384, 16385, 65792, 100000, 131072])
        if level >= 11:
            todo = [t for t in todo if len(t[1]) > 16384]
    for name, data in todo:
        exp = oracle_compress(data, level)
        got = hostsim_compress(data, level)
        assert got == exp, (name, level, exp if isinstance(exp, int) else len(exp), got if isinstance(got, int) else len(got))


@pytest.mark.parametrize("checksum,content_size", [(True, True), (False, False), (True, False)])
def test_hostsim_frame_flags_match_oracle(checksum, content_size):
    from tests.oracle_util import hostsim_compress_flags, oracle_compress_flags
    for name, data in cases.special_cases()[:3] + cases.corpus_cases(4) + cases.edge_cases(classes=(0,), sizes=[0, 1, 7, 255, 256, 1000, 65791, 65792, 131072]):
        for level in (3, 6):
            exp = oracle_compress_flags(data, level, checksum, content_size)
            assert hostsim_compress_flags(data, level, checksum, content_size) == exp, (name, level)
            if not isinstance(exp, int):
                assert hostsim_decompress(exp, len(data)) == data


def test_hostsim_decoder_on_golden_fixtures():
    man = json.loads((GOLDEN / "manifest.json").read_text())
    from tests.golden.make_golden import regenerate_input
    for e in man["oneshot"]:
        data = regenerate_input(e["input"])
        assert hostsim_decompress((GOLDEN / e["file"]).read_bytes(), len(data)) == data, e["file"]
    for e in man["decode_only"]:
        out = hostsim_decompress((GOLDEN / e["file"]).read_bytes(), e["size"])
        assert not isinstance(out, int) and hashlib.sha256(out).hexdigest() == e["sha256"], e["file"]
    for e in man["errors"]:
        assert hostsim_decompress((GOLDEN / e["file"]).read_bytes(), e["cap"]) == -e["code"], e["file"]


def test_hostsim_decoder_reference_goldens():
    for name in ["xml-1.zst", "xml-3.zst", "xml-6.zst", "xml-9.zst", "xml-1-sized.zst", "xml-advanced.zst"]:
        assert is_xml_sample(hostsim_decompress(xml_frame(name), SAMPLE)), name


def test_hostsim_decoder_matches_oracle_on_corruptions():
    import numpy as np
    from zstd_jni_b200 import corpus
    rng = np.random.default_rng(11)
    for idx in (0, 1, 2, 4, 5):
        data = corpus.chunk(idx)[:40000].tobytes()
        z = bytearray(oracle_compress(data, 3))
        for _ in range(40):
            zz = bytearray(z)
            k = int(rng.integers(0, len(zz)))
            zz[k] ^= 1 << int(rng.integers(0, 8))
            a = oracle_decompress(bytes(zz), len(data)); b = hostsim_decompress(bytes(zz), len(data))
            assert a == b, (idx, k, a if isinstance(a, int) else "ok", b if isinstance(b, int) else "ok")


def test_hostsim_decodes_reference_streams():
    """The reference's streaming path with checksums, over the 256 KB sample of `xml` (tests/golden/xml)."""
    for level in (3, 9):
        assert is_xml_sample(hostsim_decompress(xml_frame(f"xml-{level}-xxh.zst"), SAMPLE)), level


@pytest.mark.parametrize("lanes", ["32", "8"])
def test_simt_emulated_warp_matches_oracle(lanes, monkeypatch):
    """The cooperative code paths (batch probing with match_any forwarding, ballots, prefix-summed bit packing,
    in-order warp execution of sequences) on the fiber-based warp emulator, 32- and 8-lane parse groups."""
    monkeypatch.setenv("ZB_EMU_PARSE_LANES", lanes)
    todo = cases.special_cases() + cases.corpus_cases(16) + cases.edge_cases(classes=(0, 4), sizes=[0, 1, 7, 8, 64, 255, 256, 1000, 5000, 16385, 65536, 100000, 131071])
    for level in (3, 1):
        for name, data in todo:
            exp = oracle_compress(data, level)
            assert emu_compress(data, level) == exp, (name, level, lanes)
            if lanes == "32":
                assert emu_decompress(exp, len(data)) == data, (name, level)


@pytest.mark.parametrize("emu", [False, True])
def test_staged_batch_decoder_matches_oracle(emu):
    """zb_decode_fast.cuh (prepare -> Huffman streams -> sequence stream -> warp execution) on the host / the
    32-lane emulator: round trips, golden streams (multi-block items fall back to the fused path) and the same
    error code as the oracle on corrupted frames, whichever stage meets the damage."""
    import numpy as np
    from tests.oracle_util import staged_decompress
    from zstd_jni_b200 import corpus
    todo = cases.special_cases() + cases.corpus_cases(16) + cases.edge_cases(classes=(0, 2, 4, 5, 7), sizes=[0, 1, 7, 8, 64, 255, 256, 1000, 5000, 16385, 65536, 100000, 131071])
    for level in (3, 1):
        for name, data in todo:
            assert staged_decompress(oracle_compress(data, level), len(data), emu) == data, (name, level)
    # a batch packs its outputs back to back: every distance of the destination from a 4- and a 16-byte boundary
    for mis in (1, 2, 3, 5, 14):
        for name, data in cases.special_cases()[:8] + cases.corpus_cases(8) + cases.edge_cases(classes=(0, 5), sizes=[1, 7, 64, 255, 5000]):
            assert staged_decompress(oracle_compress(data, 3), len(data), emu, mis) == data, (name, mis)
    man = json.loads((GOLDEN / "manifest.json").read_text())
    for e in man["decode_only"] + man["errors"]:
        blob = (GOLDEN / e["file"]).read_bytes(); cap = e.get("size", e.get("cap"))
        assert staged_decompress(blob, cap, emu) == oracle_decompress(blob, cap), e["file"]
    rng = np.random.default_rng(21 + emu)
    for idx in (0, 1, 2, 4, 5, 7, 15, 23):
        data = corpus.chunk(idx)[:60000].tobytes(); z = oracle_compress(data, 3)
        for _ in range(40 if emu else 120):
            zz = bytearray(z); k = int(rng.integers(0, len(zz))); zz[k] ^= 1 << int(rng.integers(0, 8))
            if rng.random() < 0.2:
                zz = zz[: int(rng.integers(1, len(zz)))]
            for cap in (len(data), len(data) - 7):
                a = oracle_decompress(bytes(zz), cap); b = staged_decompress(bytes(zz), cap, emu)
                assert a == b, (idx, k, cap, a if isinstance(a, int) else "ok", b if isinstance(b, int) else "ok")


def test_randomised_levels_and_sizes():
    """Seeded fuzz over every supported level and input shape: kernel source (1 lane and 32-lane emulator) == oracle
    == compiled reference (or what it returned, tests/golden/reference_results.json)."""
    import numpy as np
    from zstd_jni_b200 import corpus
    from tests.oracle_util import ref_compress
    rng = np.random.default_rng(4242)

    def make(kind, n):
        if kind == 0:
            return corpus.chunk(int(rng.integers(0, 64))).tobytes()[:n]
        if kind == 1:
            a = np.resize(rng.integers(0, 256, int(rng.integers(3, 300)), dtype=np.uint8), n).copy()
            k = int(n * rng.random() * 0.05)
            if k:
                a[rng.integers(0, n, k)] = rng.integers(0, 256, k, dtype=np.uint8)
            return a.tobytes()
        if kind == 2:
            return rng.integers(0, int(rng.integers(2, 40)), n, dtype=np.uint8).tobytes()
        parts, left = [], n
        while left > 0:
            ln = min(left, int(rng.integers(1, 20000)))
            parts.append(make(int(rng.integers(0, 3)), ln)); left -= ln
        return b"".join(parts)

    levels = [-7, -1, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12]
    for it in range(48):
        n = int(rng.choice([rng.integers(0, 300), rng.integers(300, 16385), rng.integers(16385, 131073), 131072]))
        data = make(int(rng.integers(0, 4)), n)
        level = int(rng.choice(levels))
        exp = oracle_compress(data, level)
        if level >= 11 and n <= 16384:
            assert exp == -40
        else:
            assert exp == ref_compress(data, level), (it, n, level)
        got = hostsim_compress(data, level) if it % 2 == 0 else emu_compress(data, level)
        assert got == exp, (it, n, level)


def test_emulated_row_parser_batches_match_oracle():
    """The full-warp forms of the row-based finder (levels 5 ... 10): skipped positions inserted 32 at a time -- lanes that hit the same
    row, rows that wrap inside one batch, the 384-position skip rule -- and rows read in one round trip.  Inputs with long runs of
    equal hashes and long matches are what reaches those paths."""
    import numpy as np
    from zstd_jni_b200 import corpus
    rng = np.random.default_rng(77)
    cases = [corpus.chunk(5)[:50000].tobytes(), corpus.chunk(7 + 8 * 2)[:40000].tobytes(), corpus.chunk(0)[:30000].tobytes()]
    z = np.zeros(50000, dtype=np.uint8); z[rng.integers(0, 50000, 30)] = 9; cases.append(z.tobytes())
    for per in (3, 33):
        b = np.tile(rng.integers(0, 256, per, dtype=np.uint8), 40000 // per + 1)[:40000].copy()
        m = rng.random(40000) < 0.01; b[m] = rng.integers(0, 256, int(m.sum()), dtype=np.uint8); cases.append(b.tobytes())
    for level in (5, 9, 10):
        for k, data in enumerate(cases):
            assert emu_compress(data, level) == oracle_compress(data, level), (level, k)


def test_decoders_never_write_outside_their_destination(tmp_path):
    """tests/hostsim/canary_fuzz.cpp: corrupted and intact frames through the fused, emulated-warp and staged decoders; the destination is
    fenced by canaries on both sides (on the GPU the neighbours are other frames' outputs)."""
    import subprocess
    src = Path(__file__).parent / "hostsim" / "canary_fuzz.cpp"
    exe = tmp_path / "canary_fuzz"
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wno-unused-function", str(src), "-o", str(exe)], check=True, cwd=str(src.parent))
    out = subprocess.run([str(exe), "11", "150"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "canary violations 0" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]

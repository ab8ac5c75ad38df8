"""tests/golden/xml/: the reference's own golden vectors (src/test/resources: `xml`, a 5.3 MB XML document, and frames of it made by
its regenerate.sh), shrunk to the first 256 KB of `xml` (two full blocks, so every frame has cross-block matches) and remade with the
compiled reference (oracle/_ref) the way regenerate.sh makes them:

    xml-L-xxh.zst        L = 1, 3, 6, 9, 15: the streaming path fed 128 KB at a time (`cat xml | zstd -L`), with a checksum;
                         xml_frame("xml-L.zst") is the same frame without it (`--no-check`), see without_checksum()
    xml-1-sized.zst      one call with the content size in the header (`zstd xml -1`, not the streaming API)
    xml-advanced.zst     one call under regenerate.sh's explicit parameters (wlog=23,slog=4,tlen=32,mml=7,strat=7,hlog=16,clog=15)
    xmlsmall, xmlsmall-sized.zst    copied as they are

Only the size and SHA-256 of the 256 KB sample are kept (xml.json).  To remake the fixtures where oracle/_ref is built:
    python -m tests.golden.make_golden_xml <reference checkout>/src/test/resources
"""
from __future__ import annotations

import hashlib
import json
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
XML_DIR = HERE / "xml"
SAMPLE = 262144
LEVELS = (1, 3, 6, 9, 15)
ADVANCED = {"windowLog": 23, "searchLog": 4, "targetLength": 32, "minMatch": 7, "strategy": 7, "hashLog": 16, "chainLog": 15}


def without_checksum(frame: bytes) -> bytes:
    """The same single frame without its content checksum: clear Content_Checksum_flag, drop the 4 trailing bytes."""
    return frame[:4] + bytes([frame[4] & ~0x04]) + frame[5:-4]


def xml_manifest() -> dict:
    return json.loads((XML_DIR / "xml.json").read_text())


def xml_frame(name: str) -> bytes:
    plain = xml_manifest()["without_checksum"].get(name)
    if plain is None:
        return (XML_DIR / name).read_bytes()
    z = without_checksum((XML_DIR / name.replace(".zst", "-xxh.zst")).read_bytes())
    assert hashlib.sha256(z).hexdigest() == plain, name          # the reference's own --no-check frame
    return z


def is_xml_sample(out, copies: int = 1) -> bool:
    """out is the 256 KB sample of `xml`, `copies` times over."""
    man = xml_manifest()["sample"]
    return isinstance(out, (bytes, bytearray)) and len(out) == copies * man["size"] and hashlib.sha256(out).hexdigest() == man["sha256"][str(copies)]


def main(resources: Path):
    sys.path.insert(0, str(HERE.parent.parent))
    import ctypes as C
    from tests.oracle_util import ERR_MAX, ref, ref_compress_flags, ref_decompress, ref_stream_compress, CPARAM_IDS
    assert ref() is not None, "oracle/_ref/libzstd-oracle.so missing: build it first (oracle/Makefile, target ref)"
    xml = (resources / "xml").read_bytes()[:SAMPLE]
    XML_DIR.mkdir(exist_ok=True)
    man = {"generator": "tests/golden/make_golden_xml.py", "reference": "libzstd " + ref().ZSTD_versionString().decode(),
           "sample": {"size": len(xml), "sha256": {str(k): hashlib.sha256(xml * k).hexdigest() for k in (1, 2)}}, "without_checksum": {}}
    for level in LEVELS:
        z = ref_stream_compress(xml, level, checksum=True)
        plain = ref_stream_compress(xml, level)
        assert without_checksum(z) == plain and ref_decompress(z, len(xml)) == xml
        (XML_DIR / f"xml-{level}-xxh.zst").write_bytes(z)
        man["without_checksum"][f"xml-{level}.zst"] = hashlib.sha256(plain).hexdigest()
    (XML_DIR / "xml-1-sized.zst").write_bytes(ref_compress_flags(xml, 1, False, True))
    R = ref()
    cctx = R.ZSTD_createCCtx()
    for k, v in ADVANCED.items():
        assert R.ZSTD_CCtx_setParameter(cctx, CPARAM_IDS[k], v) <= ERR_MAX
    out = C.create_string_buffer(len(xml) + 65536)
    n = R.ZSTD_compress2(cctx, out, len(out), xml, len(xml))
    R.ZSTD_freeCCtx(cctx)
    assert n <= ERR_MAX
    (XML_DIR / "xml-advanced.zst").write_bytes(out.raw[:n])
    for name in ("xmlsmall", "xmlsmall-sized.zst"):
        (XML_DIR / name).write_bytes((resources / name).read_bytes())
    (XML_DIR / "xml.json").write_text(json.dumps(man, indent=1) + "\n")
    print(sum(f.stat().st_size for f in XML_DIR.iterdir()), "bytes in", XML_DIR)


if __name__ == "__main__":
    main(Path(sys.argv[1]))

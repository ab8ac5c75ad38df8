"""Explicit compression parameters (SURVEY.md section 8a.1: ZSTD_getCParams_internal + ZSTD_adjustCParams_internal with the
overrides of ZSTD_getCParamsFromCCtxParams, N/compress/zstd_compress.c:1623-1651): J/ZstdCompressCtx.setWindowLog / setHashLog /
setChainLog / setSearchLog / setMinMatch / setTargetLength / setStrategy.  Frames must be the reference's bytes, or the call
must refuse (window smaller than the input, optimal-parser strategies) -- never different bytes.

CPU: kernel source on the host / emulator vs tests/golden/cparams.json (made by the compiled reference) and a random
sweep against the reference itself (or what it returned, tests/golden/reference_results.json).  GPU (-m gpu): the same through the C ABI.
"""
import hashlib
import json
import random
from pathlib import Path

import pytest

from tests.golden.make_golden import regenerate_input
from tests.oracle_util import hostsim_compress_params, hostsim_decompress, ref_compress_params

GOLDEN = json.loads((Path(__file__).parent / "golden" / "cparams.json").read_text())["cases"]


def _check(e, z):
    if e["supported"]:
        assert not isinstance(z, int) and len(z) == e["size"] and hashlib.sha256(z).hexdigest() == e["sha256"], (e["input"], e["level"], e["params"])
    else:
        assert z == -40, (e["input"], e["level"], e["params"], z if isinstance(z, int) else len(z))


def test_hostsim_cparams_match_golden():
    for e in GOLDEN:
        data = regenerate_input(e["input"])
        z = hostsim_compress_params(data, e["level"], e["params"])
        _check(e, z)
        if e["supported"]:
            assert hostsim_decompress(z, len(data)) == data


def test_emulated_warp_cparams_match_golden():
    for e in GOLDEN[::7]:
        _check(e, hostsim_compress_params(regenerate_input(e["input"]), e["level"], e["params"], emu=True))


def test_hostsim_cparams_random_sweep_vs_reference():
    from zstd_jni_b200 import corpus
    rnd = random.Random(5)
    inputs = [corpus.chunk(i).tobytes() for i in (0, 1, 4, 5)] + [corpus.chunk(1)[:20000].tobytes(), corpus.chunk(2)[:5000].tobytes(), corpus.chunk(3)[:70000].tobytes()]
    for _ in range(40):
        data = rnd.choice(inputs)
        level = rnd.choice([1, 3, 4, 6, 9, -2])
        params = {k: rnd.randint(*rng) for k, rng in (("windowLog", (17, 24)), ("hashLog", (6, 22)), ("chainLog", (6, 22)), ("searchLog", (1, 8)), ("minMatch", (3, 7)),
                                                      ("targetLength", (0, 150)), ("strategy", (1, 6))) if rnd.random() < 0.4}
        assert hostsim_compress_params(data, level, params) == ref_compress_params(data, level, params), (len(data), level, params)


def test_parameter_bounds_host_side():
    """ZSTD_CCtx_setParameter bounds (ZSTD_cParam_getBounds): no GPU involved."""
    from zstd_jni_b200 import _native as N
    L = N.lib()
    c = L.ZSTD_createCCtx()
    try:
        for pid, lo, hi in ((101, 10, 31), (102, 6, 30), (103, 6, 30), (104, 1, 30), (105, 3, 7), (106, 0, 131072), (107, 1, 9)):
            assert L.ZSTD_CCtx_setParameter(c, pid, lo) == lo and L.ZSTD_CCtx_setParameter(c, pid, hi) == hi and L.ZSTD_CCtx_setParameter(c, pid, 0) == 0
            assert N.error_code(L.ZSTD_CCtx_setParameter(c, pid, hi + 1)) == 42
            if lo > 0:
                assert N.error_code(L.ZSTD_CCtx_setParameter(c, pid, lo - 1 if lo > 1 else -1)) == 42
    finally:
        L.ZSTD_freeCCtx(c)


# ------------------------------------------------------------------------------------------------ GPU
_SETTERS = {"windowLog": "setWindowLog", "hashLog": "setHashLog", "chainLog": "setChainLog", "searchLog": "setSearchLog", "minMatch": "setMinMatch",
            "targetLength": "setTargetLength", "strategy": "setStrategy"}


@pytest.mark.gpu
def test_gpu_compress_ctx_setters_match_golden():
    from zstd_jni_b200.zstd import Zstd, ZstdCompressCtx, ZstdException
    from tests.oracle_util import oracle_compress
    with ZstdCompressCtx() as c:
        for e in GOLDEN:
            data = regenerate_input(e["input"])
            c.reset()
            c.setLevel(e["level"])
            for k, v in e["params"].items():
                getattr(c, _SETTERS[k])(v)
            if e["supported"]:
                z = c.compress(data)
                _check(e, z)
                assert Zstd.decompress(z, len(data)) == data
            else:
                with pytest.raises(ZstdException) as ei:
                    c.compress(data)
                assert ei.value.getErrorCode() == 40
        # parameters persist across calls of a context and are dropped by reset() (ZSTD_reset_session_and_parameters)
        data = regenerate_input({"kind": "corpus", "index": 1, "size": 131072})
        c.reset()
        c.setLevel(3).setHashLog(12)
        a = c.compress(data)
        assert a == c.compress(data) and a != oracle_compress(data, 3)
        c.setHashLog(0)
        assert c.compress(data) == oracle_compress(data, 3)
        c.setStrategy(8)                                   # btultra: accepted as a value, but no GPU parser
        with pytest.raises(ZstdException) as ei:
            c.compress(data)
        assert ei.value.getErrorCode() == 40
        c.reset()
        assert c.compress(data) == oracle_compress(data, 3)


@pytest.mark.gpu
def test_gpu_batch_option_cparams_and_reference_sweep():
    from zstd_jni_b200 import corpus
    from zstd_jni_b200.zstd import ZstdBatchContext
    from tests.oracle_util import oracle_compress
    chunks = [corpus.chunk(i).tobytes() for i in range(16)] + [corpus.chunk(1)[:20000].tobytes(), corpus.chunk(2)[:5000].tobytes(), b"", b"abcdefg" * 3]
    rnd = random.Random(11)
    with ZstdBatchContext(0) as ctx:
        for trial in range(6):
            level = rnd.choice([1, 3, 5, 9])
            params = {k: rnd.randint(*rng) for k, rng in (("windowLog", (17, 24)), ("hashLog", (6, 22)), ("chainLog", (6, 22)), ("searchLog", (1, 8)), ("minMatch", (3, 7)),
                                                          ("targetLength", (0, 150)), ("strategy", (1, 6))) if rnd.random() < 0.4} or {"hashLog": 10}
            for k in _SETTERS:
                ctx.setOption("c_" + k, params.get(k, 0))
            frames = ctx.compressBatch(chunks, level)
            assert ctx.decompressBatch(frames, [len(x) for x in chunks]) == chunks
            for x, f in zip(chunks, frames):
                assert f == ref_compress_params(x, level, params), (trial, level, params, len(x))
        ctx.setOption("c_windowLog", 15)                   # a window smaller than the input: refused per frame, small inputs still compress
        for k in _SETTERS:
            if k != "windowLog":
                ctx.setOption("c_" + k, 0)
        out = ctx.compressBatch(chunks[14:], 3, raise_on_error=False)
        assert out[0] == -40 and out[1] == -40 and not isinstance(out[2], int) and not isinstance(out[3], int)
        assert out[2] == ref_compress_params(chunks[16], 3, {"windowLog": 15}) and out[3] == ref_compress_params(chunks[17], 3, {"windowLog": 15})
        ctx.setOption("c_windowLog", 0)
        assert ctx.compressBatch(chunks[:2], 3) == [oracle_compress(x, 3) for x in chunks[:2]]
        with pytest.raises(KeyError):
            ctx.setOption("c_minMatch", 8)

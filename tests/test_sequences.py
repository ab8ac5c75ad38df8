"""The match finder behind the reference's sequence-level plug points (SURVEY.md section 8f.4):
ZSTD_generateSequences (N/compress/zstd_compress.c:3520-3553) and the block-level external sequence producer
(ZSTD_sequenceProducer_F, N/zstd.h:2820-2900; J/SequenceProducer.java).

CPU: the kernel source (parse_stage + export_sequences) on the host / on the 32-lane emulator against the golden
fixtures made by the compiled reference (tests/golden/sequences.json) and against the
reference itself (or what it returned, tests/golden/reference_results.json); where oracle/_ref is built, the producer contract is
exercised by plugging the host instantiation into the reference's libzstd.
GPU (-m gpu): the same through the C ABI, and the real zstdb200_sequenceProducer registered in the reference's libzstd.
"""
import ctypes as C
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

from tests import cases
from tests.golden.make_golden import regenerate_input
from tests.oracle_util import ERR_MAX, hostsim, hostsim_generate_sequences, ref, ref_decompress, ref_generate_sequences, same

GOLDEN = json.loads((Path(__file__).parent / "golden" / "sequences.json").read_text())["cases"]
PRODUCER_F = C.CFUNCTYPE(C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_size_t)
ZSTD_c_validateSequences = 1012          # ZSTD_c_experimentalParam12 (N/zstd.h)
ZSTD_c_enableSeqProducerFallback = 1017  # ZSTD_c_experimentalParam17


def _digest(seqs) -> str:
    return hashlib.sha256(np.ascontiguousarray(seqs, dtype="<u4").tobytes()).hexdigest()


def _check_valid_parse(seqs, data: bytes):
    """The validity conditions of N/zstd.h:2862-2872 plus: replaying the sequences regenerates the block."""
    assert seqs[-1][0] == 0 and seqs[-1][2] == 0
    out = bytearray()
    pos = 0
    for off, ll, ml, _rep in seqs.tolist():
        out += data[pos:pos + ll]
        pos += ll
        if ml:
            assert ml >= 3 and 0 < off <= len(out)
            for _ in range(ml):
                out.append(out[-off])
            pos += ml
    assert bytes(out) == data


def test_hostsim_sequences_match_golden():
    for e in GOLDEN:
        data = regenerate_input(e["input"])
        assert hashlib.sha256(data).hexdigest() == e["input_sha256"]
        got = hostsim_generate_sequences(data, e["level"])
        assert not isinstance(got, int) and got.shape[0] == e["count"] and _digest(got) == e["sha256"], (e["input"], e["level"])


def test_emulated_warp_sequences_match_golden():
    todo = [e for e in GOLDEN if e["level"] in (3, 1)][::3]
    for e in todo:
        data = regenerate_input(e["input"])
        got = hostsim_generate_sequences(data, e["level"], emu=True)
        assert not isinstance(got, int) and _digest(got) == e["sha256"], (e["input"], e["level"])


def test_hostsim_sequences_match_reference_and_replay():
    for level in (3, 1, 7):
        for name, data in cases.special_cases()[:6] + cases.corpus_cases(8) + cases.edge_cases(classes=(0, 5), sizes=[7, 8, 9, 64, 1000, 16385, 70000, 131072]):
            exp = ref_generate_sequences(data, level)
            got = hostsim_generate_sequences(data, level)
            assert not isinstance(exp, int) and not isinstance(got, int), (name, level)
            assert same(exp, got), (name, level)
            if level == 3:
                _check_valid_parse(got, data)


def _compress_with_producer(fn_ptr, state, data: bytes, level: int):
    R = ref()
    cctx = R.ZSTD_createCCtx()
    try:
        assert R.ZSTD_CCtx_setParameter(cctx, 100, level) <= ERR_MAX
        assert R.ZSTD_CCtx_setParameter(cctx, ZSTD_c_validateSequences, 1) <= ERR_MAX
        assert R.ZSTD_CCtx_setParameter(cctx, ZSTD_c_enableSeqProducerFallback, 0) <= ERR_MAX
        R.ZSTD_registerSequenceProducer(cctx, state, fn_ptr)
        cap = R.ZSTD_compressBound(len(data))
        out = C.create_string_buffer(cap)
        n = R.ZSTD_compress2(cctx, out, cap, data, len(data))
        return out.raw[:n] if n <= ERR_MAX else -((1 << 64) - n)
    finally:
        R.ZSTD_freeCCtx(cctx)


def _multi_block_input():
    from zstd_jni_b200 import corpus
    return b"".join(corpus.chunk(i).tobytes() for i in (1, 9, 5, 17))[:450000]


def test_host_instantiation_is_a_valid_sequence_producer():
    """The record layout and the block-delimiter convention are what libzstd's external-sequence path accepts
    (ZSTD_c_validateSequences on, no fallback): kernel source on the host behind a ctypes callback."""
    if ref() is None:
        pytest.skip("oracle/_ref not built on this machine")
    H = hostsim()
    calls = []

    def producer(state, out_seqs, cap, src, src_size, dict_, dict_size, level, window):
        n = H.zbh_generate_sequences(out_seqs, cap, C.string_at(src, src_size), src_size, level, 0)
        calls.append((src_size, n))
        return n

    cb = PRODUCER_F(producer)
    data = _multi_block_input()
    z = _compress_with_producer(C.cast(cb, C.c_void_p), None, data, 3)
    assert not isinstance(z, int), z
    assert [c[0] for c in calls] == [131072, 131072, 131072, 450000 - 3 * 131072]
    assert ref_decompress(z, len(data)) == data
    assert len(z) < len(data) // 4


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_gpu_generate_sequences_matches_golden_and_reference():
    from zstd_jni_b200.zstd import ZstdBatchContext
    with ZstdBatchContext(0) as ctx:
        for level in sorted({e["level"] for e in GOLDEN}):
            todo = [e for e in GOLDEN if e["level"] == level]
            blocks = [regenerate_input(e["input"]) for e in todo]
            before = ctx.kernelLaunches()
            got = ctx.generateSequences(blocks, level)
            assert ctx.kernelLaunches() >= before + 2          # k_parse + k_seq_export at least
            for e, g, data in zip(todo, got, blocks):
                assert not isinstance(g, int) and g.shape[0] == e["count"] and _digest(g) == e["sha256"], (e["input"], level)
        todo = cases.special_cases() + cases.corpus_cases(24) + cases.edge_cases(classes=(0, 2, 4, 5, 7))
        blocks = [d for _, d in todo]
        for level in (3, 1, 5):
            got = ctx.generateSequences(blocks, level, raise_on_error=False)
            for (name, data), g in zip(todo, got):
                exp = ref_generate_sequences(data, level)
                if len(data) == 0:
                    assert not isinstance(g, int) and g.shape[0] == 0, name
                elif isinstance(exp, int):
                    assert g == exp == -106, (name, level, g, exp)          # srcSize < 7: sequenceProducer_failed
                else:
                    assert same(exp, g), (name, level)


@pytest.mark.gpu
def test_gpu_generate_sequences_capacity_and_size_errors():
    from zstd_jni_b200 import _native as N, corpus
    L = N.lib()
    ctx = L.zstdb200_create(0)
    assert ctx
    try:
        data = corpus.chunk(1).tobytes()
        src = (C.c_void_p * 2)(C.cast(C.c_char_p(data), C.c_void_p), C.cast(C.c_char_p(data), C.c_void_p))
        ssz = (C.c_size_t * 2)(len(data), 1000)
        outs = [np.zeros((8, 4), dtype=np.uint32), np.zeros((400, 4), dtype=np.uint32)]
        dst = (C.c_void_p * 2)(outs[0].ctypes.data, outs[1].ctypes.data)
        cap = (C.c_size_t * 2)(8, 400)
        nb = (C.c_size_t * 2)()
        r = L.zstdb200_generate_sequences(ctx, 3, 2, src, ssz, dst, cap, nb)
        assert N.error_code(r) == 70 and N.error_code(nb[0]) == 70 and not N.is_error(nb[1]) and nb[1] >= 1
        _check_valid_parse(outs[1][: nb[1]], data[:1000])
        ssz[0] = 131073
        r = L.zstdb200_generate_sequences(ctx, 3, 2, src, ssz, dst, cap, nb)
        assert N.error_code(r) == 72
        r = L.zstdb200_generate_sequences(ctx, 19, 2, src, ssz, dst, cap, nb)
        assert N.error_code(r) == 40                              # optimal-parser levels have no GPU parser
    finally:
        L.zstdb200_free(ctx)


@pytest.mark.gpu
def test_gpu_sequence_producer_inside_reference_libzstd():
    """J/SequenceProducer.java contract: function pointer + state registered with the reference's own libzstd, which
    keeps the frame / block loop / entropy stage and calls the GPU for the match finding of every block."""
    if ref() is None:
        pytest.skip("oracle/_ref not built on this machine")
    from zstd_jni_b200 import _native as N
    from zstd_jni_b200.zstd import B200SequenceProducer
    prod = B200SequenceProducer(0)
    state = prod.createState()
    try:
        launches0 = N.lib().zstdb200_kernel_launches(state)
        for level, data in ((3, _multi_block_input()), (1, _multi_block_input()[:200001]), (3, cases.corpus_cases(3)[2][1]), (5, _multi_block_input()[:140000])):
            z = _compress_with_producer(prod.getFunctionPointer(), state, data, level)
            assert not isinstance(z, int), (level, z)
            assert ref_decompress(z, len(data)) == data
        assert N.lib().zstdb200_kernel_launches(state) > launches0
        # direct calls: error paths of the producer itself
        out = np.zeros((64, 4), dtype=np.uint32)
        f = N.lib().zstdb200_sequenceProducer
        small = b"abcabc"
        assert f(state, out.ctypes.data, 64, small, 6, None, 0, 3, 1 << 17) == 1 and out[0].tolist() == [0, 6, 0, 0]
        assert f(state, out.ctypes.data, 64, small, 6, small, 6, 3, 1 << 17) == (1 << 64) - 1      # dictionaries are not supported
        assert f(state, out.ctypes.data, 64, small * 100, 600, None, 0, 22, 1 << 17) == (1 << 64) - 1   # no GPU parser for level 22
        assert f(None, out.ctypes.data, 64, small, 6, None, 0, 3, 1 << 17) == (1 << 64) - 1
    finally:
        prod.freeState(state)

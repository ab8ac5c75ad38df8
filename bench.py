#!/usr/bin/env python
"""bench.py -- the headline benchmark (BASELINE.json: uncompressed GB/s, level-3 compress + decompress).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--chunks C] [--level L] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

A *step* is one pass of the hot path over one batch: every rank compresses its shard of C 128 KB chunks
(level 3, one frame per chunk, sizes scanned and frames concatenated on the device) and decompresses the
resulting stream back.  Default workload = BASELINE.json configs[1]: a 1 GiB synthetic Silesia-mix corpus
(8192 x 131072 B, seed 20240901) on one B200.  With N GPUs every rank gets its own 8192-chunk shard (weak
scaling); frames are independent so there is no data-path exchange, only an all_gather of the per-frame sizes
(the global stream index) and the timing reduction.

Printed (rank 0, one JSON line): value = uncompressed bytes taken through compress+decompress per second with
inputs resident in HBM (CUDA events on the launching stream, max over ranks); e2e = the same through the
host-memory C-ABI calls (pinned host buffers, H2D + kernels + D2H timed); roofline = dominant timed entry vs the
measured HBM peak -- the two compression stages run overlapped (k_entropy is a programmatic dependent of k_parse), so they
are ONE entry "k_parse+k_entropy" in kernel_ms; their separate times come from a short serialized pass outside the timed
region (kernel_ms_serialized); cpu_baseline = the reference's own libzstd (oracle/_ref) on this box's host cores.
`--impl reference` times only that CPU path with all host threads and prints the same line shape.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
CHUNK = 131072
METRIC = "uncompressed GB/s, level-3 compress + decompress round trip (zstd, 128 KB frames)"


# ----------------------------------------------------------------------------- CPU reference arm
def _cpu_lib():
    """The reference's own C sources compiled in place (kind 'reference'), else the plain-C port."""
    ref = ROOT / "oracle" / "_ref" / "libzstd-oracle.so"
    if ref.exists():
        L = C.CDLL(str(ref))
        for n, a in (("ZSTD_compress2", [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
                     ("ZSTD_decompressDCtx", [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
                     ("ZSTD_CCtx_setParameter", [C.c_void_p, C.c_int, C.c_int]), ("ZSTD_freeCCtx", [C.c_void_p]), ("ZSTD_freeDCtx", [C.c_void_p])):
            getattr(L, n).argtypes = a
            getattr(L, n).restype = C.c_size_t
        L.ZSTD_createCCtx.restype = C.c_void_p
        L.ZSTD_createDCtx.restype = C.c_void_p
        return L, "reference"
    port = ROOT / "oracle" / "libzso.so"
    if not port.exists():
        subprocess.run(["make", "-s", "-C", str(ROOT / "oracle"), "libzso.so"], check=True)
    L = C.CDLL(str(port))
    L.zso_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int]
    L.zso_compress.restype = C.c_size_t
    L.zso_decompress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    L.zso_decompress.restype = C.c_size_t
    return L, "port"


class CpuRoundTrip:
    """Per-call path of N/jni_fast_zstd.c:633-635,825-826 minus JNI: one ctx per thread, static partition of the
    chunks, ZSTD_compress2 then ZSTD_decompressDCtx.  ctypes releases the GIL so the threads run in parallel.
    Buffers are allocated and touched once so that page faults stay out of the timed region."""

    def __init__(self, data: np.ndarray, level: int, threads: int):
        self.L, self.kind = _cpu_lib()
        self.data, self.level, self.threads = data, level, threads
        n = data.shape[0]
        self.bound = CHUNK + (CHUNK >> 8) + 64
        self.comp = np.zeros((n, self.bound), dtype=np.uint8)
        self.sizes = np.zeros(n, dtype=np.int64)
        self.back = np.zeros_like(data)
        self.parts = [range(t, n, threads) for t in range(threads)]
        self.src_ptr = [int(data[i].ctypes.data) for i in range(n)]
        self.comp_ptr = [int(self.comp[i].ctypes.data) for i in range(n)]
        self.back_ptr = [int(self.back[i].ctypes.data) for i in range(n)]
        self.pool = ThreadPoolExecutor(threads)

    def _c(self, idx):
        L, size, bound, level = self.L, self.data.shape[1], self.bound, self.level
        if self.kind == "reference":
            cctx = L.ZSTD_createCCtx()
            L.ZSTD_CCtx_setParameter(cctx, 100, level)
            for i in idx:
                self.sizes[i] = L.ZSTD_compress2(cctx, self.comp_ptr[i], bound, self.src_ptr[i], size)
            L.ZSTD_freeCCtx(cctx)
        else:
            for i in idx:
                self.sizes[i] = L.zso_compress(self.comp_ptr[i], bound, self.src_ptr[i], size, level)

    def _d(self, idx):
        L, size = self.L, self.data.shape[1]
        if self.kind == "reference":
            dctx = L.ZSTD_createDCtx()
            for i in idx:
                L.ZSTD_decompressDCtx(dctx, self.back_ptr[i], size, self.comp_ptr[i], int(self.sizes[i]))
            L.ZSTD_freeDCtx(dctx)
        else:
            for i in idx:
                L.zso_decompress(self.back_ptr[i], size, self.comp_ptr[i], int(self.sizes[i]))

    def run(self):
        """-> (t_compress, t_decompress, compressed_bytes)"""
        t0 = time.perf_counter(); list(self.pool.map(self._c, self.parts)); t1 = time.perf_counter()
        list(self.pool.map(self._d, self.parts)); t2 = time.perf_counter()
        return t1 - t0, t2 - t1, int(self.sizes.sum())

    def check(self):
        assert np.array_equal(self.back, self.data), "CPU reference round trip failed"


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampled every 200 ms while the timed region runs (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.samples = []
        self.proc = None
        self.index = index

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for s in self.samples if len(s) >= 7 for k in range(4) if s[3 + k].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chunks", type=int, default=8192, help="128 KB chunks per GPU (8192 = 1 GiB, BASELINE.json configs[1])")
    ap.add_argument("--level", type=int, default=3)
    ap.add_argument("--cpu-chunks", type=int, default=0, help="chunks in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the sub-records (levels, configs[3], configs[4])")
    ap.add_argument("--strong", action="store_true", help="also run the strong-scaling data-plane record at N = 1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed on rank 0 to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    from zstd_jni_b200 import corpus

    config = {"workload": f"{args.chunks} x {CHUNK} B synthetic Silesia-mix chunks per GPU (seed {corpus.SEED}), level {args.level}, one frame per chunk",
              "chunks_per_gpu": args.chunks, "chunk_bytes": CHUNK, "level": args.level, "cache": "inputs_larger_than_L2 (1 GiB working set per pass vs 126 MB L2)",
              "parallelism": f"frames sharded over {args.gpus} GPU(s), no data-path collective"}

    if args.impl == "reference":
        if rank != 0:
            return
        threads = host_threads()
        # bounded sample of the same workload: the first n chunks of the corpus, sized for a few seconds per step
        n = args.cpu_chunks or min(args.chunks, max(512, 128 * threads))
        data = corpus.corpus(n)
        cpu = CpuRoundTrip(data, args.level, threads)
        for _ in range(max(1, args.warmup)):
            cpu.run()
        cpu.check()
        times = []
        for _ in range(args.steps):
            tc, td, csize = cpu.run()
            times.append((tc, td))
        kind = cpu.kind
        tc = float(np.median([t[0] for t in times])); td = float(np.median([t[1] for t in times]))
        U = data.size
        val = U / (tc + td) / 1e9
        print(json.dumps({"metric": METRIC, "value": val, "unit": "GB/s", "impl": "reference", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": (tc + td) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                          "config": config, "compress_gbs": U / tc / 1e9, "decompress_gbs": U / td / 1e9, "ratio": U / csize,
                          "cpu_baseline": {"value": val, "unit": "GB/s", "cores": threads, "kind": kind, "cpu": cpu_model(),
                                           "sample": f"first {n} chunks ({U / 2**20:.0f} MiB) of the corpus, {threads} threads, ctx per thread"},
                          "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line (NCCL prints its version banner there)
    import torch
    import torch.distributed as dist
    from zstd_jni_b200 import _native
    from zstd_jni_b200.zstd import ZstdBatchContext
    from zstd_jni_b200 import sharding
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the product has no CPU fallback); use --impl reference for the CPU arm"
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL prints its version banner on stdout when the first communicator comes up; the contract is ONE JSON line there, so
        # stdout points at stderr until the communicator exists
        sys.stdout.flush(); saved = os.dup(1); os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier(); torch.cuda.synchronize()
        finally:
            sys.stdout.flush(); os.dup2(saved, 1); os.close(saved)
    L = _native.lib()
    ctx = ZstdBatchContext(local)
    n = args.chunks
    dev = torch.device("cuda", local)
    data = corpus.corpus(n, start=rank * n)                                   # this rank's shard
    h_src = torch.from_numpy(data.reshape(-1)).pin_memory()
    d_src = h_src.to(dev)
    d_off = torch.arange(0, (n + 1) * CHUNK, CHUNK, dtype=torch.int64, device=dev)
    stride = (L.ZSTD_compressBound(CHUNK) + 32 + 63) // 64 * 64
    d_slots = torch.empty(n * stride, dtype=torch.uint8, device=dev)
    d_sizes = torch.zeros(n, dtype=torch.int64, device=dev)
    d_out = torch.empty(n * stride, dtype=torch.uint8, device=dev)
    d_ooff = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    d_back = torch.empty(n * CHUNK, dtype=torch.uint8, device=dev)
    d_res = torch.zeros(n, dtype=torch.int64, device=dev)
    index = {}
    stream = torch.cuda.Stream(device=dev)
    st = stream.cuda_stream
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def check(r):
        if _native.is_error(r):
            raise RuntimeError(f"C ABI error {L.ZSTD_getErrorName(r).decode()} / {L.zstdb200_last_error().decode()}")

    def step(events=None):
        """compress (+scan+concat) then decompress, all on `stream`; optional per-kernel events"""
        if events: events[0].record(stream)
        check(L.zstdb200_compress_device(ctx.handle, args.level, n, d_src.data_ptr(), d_off.data_ptr(), d_slots.data_ptr(), stride, d_sizes.data_ptr(), st))
        if events: events[1].record(stream)
        check(L.zstdb200_compact_device(ctx.handle, n, d_slots.data_ptr(), stride, d_sizes.data_ptr(), d_out.data_ptr(), d_ooff.data_ptr(), st))
        if world > 1:
            # global stream index (8 B x frames over NCCL); the only exchange on this path
            index["offsets"] = sharding.global_offsets(sharding.gather_sizes(d_sizes, world * n))
        if events: events[2].record(stream)
        check(L.zstdb200_decompress_device(ctx.handle, n, d_out.data_ptr(), d_ooff.data_ptr(), d_back.data_ptr(), d_off.data_ptr(), d_res.data_ptr(), st))
        if events: events[3].record(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step()
        barrier()
        assert torch.equal(d_back, d_src) and bool((d_res == CHUNK).all()), "device round trip mismatch"
        csize = int(d_sizes.sum().item())
        sampler = ClockSampler(local); sampler.start()
        launches0 = ctx.kernelLaunches()
        ctx.setOption("timing", 1)          # the library brackets every kernel with CUDA events on its launching stream
        ctx.kernelTimes()
        evs = [[ev() for _ in range(4)] for _ in range(args.steps)]
        barrier()
        t_begin, t_end = ev(), ev()
        t_begin.record(stream)
        for k in range(args.steps):
            step(evs[k])
        t_end.record(stream)
        barrier()
        launches = ctx.kernelLaunches() - launches0
        ktimes = ctx.kernelTimes()
        clocks = sampler.stop()
        if args.dump_outputs and rank == 0:
            dump_outputs(Path(args.dump_outputs), n, d_sizes, d_ooff, d_out, d_back, d_res)
        # The entropy stage runs beside the parse (one timed entry, "k_parse+k_entropy"); a short pass with the two serialized gives the
        # stage times on their own -- reported as such, not part of the timed region.
        ctx.setOption("entropy_overlap", 0)
        for _ in range(3):
            step()
        barrier()
        ktimes_serial = ctx.kernelTimes()
        ctx.setOption("entropy_overlap", 1)
        ctx.setOption("timing", 0)
    total_ms = t_begin.elapsed_time(t_end)
    k_comp = float(np.mean([e[0].elapsed_time(e[1]) for e in evs])); k_pack = float(np.mean([e[1].elapsed_time(e[2]) for e in evs])); k_dec = float(np.mean([e[2].elapsed_time(e[3]) for e in evs]))
    tms = torch.tensor([total_ms, k_comp, k_pack, k_dec], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    total_ms, k_comp, k_pack, k_dec = [float(x) for x in tms.tolist()]
    U = n * CHUNK
    ms_per_step = total_ms / args.steps
    value = world * U / (ms_per_step * 1e-3) / 1e9

    # ---- end to end through the host-memory C ABI (pinned buffers; H2D + kernels + D2H inside the timed region).
    # The asynchronous begin/end pair keeps batches in flight on four work sets: while step k is in the kernels, the input of
    # step k+1 rides in and the results of step k-1 ride out.  Every step still moves its whole input H2D and its whole result D2H
    # inside the timed region; the stream decompressed in step k is the one step k compressed.
    numa = sharding.bind_to_gpu_numa(local)                      # pinned buffers next to this rank's GPU
    h_stream = [torch.empty(n * stride, dtype=torch.uint8).pin_memory() for _ in range(2)]
    h_back = [torch.empty(n * CHUNK, dtype=torch.uint8).pin_memory() for _ in range(2)]
    fsz = [(C.c_size_t * n)() for _ in range(2)]; dsz = [(C.c_size_t * n)() for _ in range(2)]
    dsz_in = (C.c_size_t * n)(*([CHUNK] * n))          # expected sizes (in)
    tot = C.c_size_t(0)
    def cb(k): check(L.zstdb200_compress_chunks_begin(ctx.handle, k % 2, args.level, h_src.data_ptr(), U, CHUNK))
    def ce(k): check(L.zstdb200_compress_chunks_end(ctx.handle, k % 2, h_stream[k % 2].data_ptr(), h_stream[k % 2].numel(), fsz[k % 2], C.byref(tot)))
    def db(k): check(L.zstdb200_decompress_frames_begin(ctx.handle, 2 + k % 2, h_stream[k % 2].data_ptr(), fsz[k % 2], n, h_back[k % 2].data_ptr(), h_back[k % 2].numel(), dsz_in))
    def de(k): check(L.zstdb200_decompress_frames_end(ctx.handle, 2 + k % 2, dsz[k % 2]))
    def e2e_run(K):
        cb(0)
        for k in range(K):
            if k + 1 < K: cb(k + 1)
            ce(k); db(k)
            if k >= 1: de(k - 1)
        de(K - 1)
        torch.cuda.synchronize()
    e2e_run(2); barrier()
    e2e_steps = args.steps                           # the pipeline fills and drains once per run (~60 ms that no step can hide)
    t0 = time.perf_counter()
    e2e_run(e2e_steps)
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    assert torch.equal(h_back[(e2e_steps - 1) % 2], h_src) and torch.equal(h_back[e2e_steps % 2], h_src), "e2e round trip mismatch"
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = world * U / float(te.item()) / 1e9
    # the synchronous pair for comparison (one batch at a time: copies and kernels add up)
    def sync_step():
        check(L.zstdb200_compress_chunks(ctx.handle, args.level, h_src.data_ptr(), U, CHUNK, h_stream[0].data_ptr(), h_stream[0].numel(), fsz[0], C.byref(tot)))
        C.memmove(dsz[0], dsz_in, C.sizeof(dsz_in))
        check(L.zstdb200_decompress_frames(ctx.handle, h_stream[0].data_ptr(), fsz[0], n, h_back[0].data_ptr(), h_back[0].numel(), dsz[0]))
    sync_step(); t0 = time.perf_counter(); sync_step(); torch.cuda.synchronize(); sync_s = time.perf_counter() - t0

    strong = strong_scaling(args, ctx, L, dev, rank, world, local, check, barrier) if (world > 1 or args.strong) else None

    if rank != 0:
        if world > 1: dist.destroy_process_group()
        return
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak = float(json.loads(peaks_path.read_text())["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak = 6650.0; peak_src = "fallback (B200_PROFILING.md 6.65 TB/s)"
    algo_bytes = U + csize                                  # SURVEY.md 8(d): uncompressed + compressed bytes of every frame in the launch
    # per-kernel averages over the timed region (rank 0), from the events the library records around every launch
    kernels = {k: v[0] for k, v in ktimes.items()}
    serial = {k: v[0] for k, v in ktimes_serial.items()}      # k_parse and k_entropy one after the other (untimed-region pass)
    PAIR = "k_parse+k_entropy"
    phases = {"compress": k_comp, "scan+compact": k_pack, "decompress": k_dec}          # API-call brackets, max over ranks
    payload = {k: v for k, v in kernels.items() if k not in ("k_order", "k_parse(estimate)", "k_dec_prepare", "k_decompress")}
    dom = max(payload, key=payload.get)
    traffic = {}
    tpath = ROOT / "profiles" / "dram_traffic.json"          # dram__bytes_read.sum + dram__bytes_write.sum per launch (ncu --set full)
    if tpath.exists():
        tj = json.loads(tpath.read_text())
        if tj.get("chunks_per_gpu") == n and tj.get("level") == args.level:
            traffic = tj.get("kernels", {})
    # algorithmic bytes per kernel (payload kernels only): what the stage has to read and write once, SURVEY.md 8(d) split by stage
    stage_bytes = {PAIR: (U + csize, "the two compression stages, overlapped: the input is read, the frames are written"),
                   "k_parse": (U, "reads the input"), "k_entropy": (U + csize, "reads the input (literals), writes the frames"),
                   "k_scan_sizes+k_compact": (2 * csize, "reads and writes the frames"), "k_dec_chains": (csize, "reads the frames' bitstreams"),
                   "k_dec_exec": (U, "writes the regenerated bytes")}
    if PAIR in kernels and "k_parse" in traffic and "k_entropy" in traffic:
        traffic = dict(traffic); traffic[PAIR] = traffic["k_parse"] + traffic["k_entropy"]
    def roof(name, nbytes, table=None):
        a = nbytes / ((table or kernels)[name] * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak, "traffic": traffic.get(name), "bytes": nbytes}
    roofline_all = {k: dict(roof(k, stage_bytes[k][0]), what=stage_bytes[k][1], timed="timed region") for k in kernels if k in stage_bytes}
    for k in ("k_parse", "k_entropy"):
        if k in serial and k not in roofline_all:
            roofline_all[k] = dict(roof(k, stage_bytes[k][0], serial), what=stage_bytes[k][1], timed="serialized pass (entropy_overlap off), outside the timed region")
    out = {"metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
           "compress_gbs": world * U / ((k_comp + k_pack) * 1e-3) / 1e9, "decompress_gbs": world * U / (k_dec * 1e-3) / 1e9, "ratio": U / csize,
           "decompress_hbm_frac": (U + csize) / (k_dec * 1e-3) / 1e9 / peak,
           "kernel_ms": kernels, "kernel_ms_serialized": {k: serial[k] for k in ("k_parse", "k_entropy") if k in serial}, "phase_ms": phases,
           "roofline": dict(roof(dom, algo_bytes), kernel=dom, peak_source=peak_src, algorithmic_bytes_per_launch=algo_bytes,
                            launches_timed=ktimes[dom][1]),
           "roofline_all": roofline_all,
           "e2e": {"value": e2e_val, "unit": "GB/s", "h2d_bytes_per_step": U + csize, "d2h_bytes_per_step": csize + U, "ms_per_step": float(te.item()) * 1e3,
                   "api": "zstdb200_compress_chunks_begin/_end + zstdb200_decompress_frames_begin/_end on 4 work sets, pinned host buffers; "
                          "every step's input goes H2D and its result D2H inside the timed region, steps overlap",
                   "steps": e2e_steps, "synchronous_ms_per_step": sync_s * 1e3, "numa": numa},
           "gpu_launches": int(launches), "clocks": clocks}
    if strong is not None:
        out["strong"] = strong
    if not args.no_cpu_baseline and world == 1:
        threads = host_threads()
        ncpu = args.cpu_chunks or min(n, max(512, 128 * threads))
        cpu = CpuRoundTrip(data[:ncpu], args.level, threads)
        cpu.run(); cpu.check()
        runs = [cpu.run() for _ in range(3)]
        tc = float(np.median([r[0] for r in runs])); td = float(np.median([r[1] for r in runs])); kind = cpu.kind
        Uc = ncpu * CHUNK
        out["cpu_baseline"] = {"value": Uc / (tc + td) / 1e9, "unit": "GB/s", "cores": threads, "kind": kind, "cpu": cpu_model(),
                               "compress_gbs": Uc / tc / 1e9, "decompress_gbs": Uc / td / 1e9,
                               "sample": f"first {ncpu} chunks ({Uc / 2**20:.0f} MiB) of the same corpus, {threads} threads, one ctx per thread"}
        # full-configuration parity: every frame the GPU wrote in the end-to-end leg against the frame the reference wrote for the same chunk
        hs = h_stream[(e2e_steps - 1) % 2].numpy(); sizes_g = np.ctypeslib.as_array(fsz[(e2e_steps - 1) % 2]).astype(np.int64)
        offs_g = np.concatenate([[0], np.cumsum(sizes_g)])
        same = 0
        for i in range(ncpu):
            sz = int(cpu.sizes[i])
            if sz == int(sizes_g[i]) and np.array_equal(cpu.comp[i, :sz], hs[offs_g[i]:offs_g[i] + sz]):
                same += 1
        out["parity"] = {"frames": ncpu, "identical": same, "against": f"{kind} (oracle/_ref libzstd 1.5.7, ZSTD_compress2 level {args.level})" if kind == "reference" else kind}
        if not args.no_extra:
            out["levels"] = levels_record(args, ctx, L, dev, n, d_src, d_off, d_slots, d_sizes, d_out, d_ooff, stride, st, stream, data, threads, check)
            out["config3_decompress_only"] = config3_record(args, ctx, L, dev, stream, st, check, threads)
            out["config4_streaming"] = config4_record(args, data, threads)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir: Path, n, d_sizes, d_ooff, d_out, d_back, d_res):
    """What a caller of the timed path receives, as float arrays (bytes and sizes are exact in them), so that two builds can be compared
    output for output: every frame size and regenerated size, and for a fixed, seeded sample of 32 chunks their frames and regenerated
    bytes (about 25 MB for the default workload, at most 34 MB; the whole round trip is checked on the device by the run itself)."""
    out_dir.mkdir(parents=True, exist_ok=True)
    offs = d_ooff.cpu().numpy()
    pick = np.sort(np.random.default_rng(0).choice(n, size=min(n, 32), replace=False))
    frames = np.concatenate([d_out[offs[i]:offs[i + 1]].cpu().numpy() for i in pick])
    back = np.concatenate([d_back[i * CHUNK:(i + 1) * CHUNK].cpu().numpy() for i in pick])
    np.save(out_dir / "frame_sizes.npy", d_sizes.cpu().numpy().astype(np.float64))
    np.save(out_dir / "decompressed_sizes.npy", d_res.cpu().numpy().astype(np.float64))
    np.save(out_dir / "sample_chunks.npy", pick.astype(np.float64))
    np.save(out_dir / "sample_frames.npy", frames.astype(np.float32))
    np.save(out_dir / "sample_decompressed.npy", back.astype(np.float32))


# ----------------------------------------------------------------------------- sub-records
def _time_ms(stream, fn, reps=3):
    import torch
    fn(); torch.cuda.synchronize()
    best = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream); fn(); e1.record(stream)
        torch.cuda.synchronize()
        best.append(e0.elapsed_time(e1))
    return float(np.median(best))


def levels_record(args, ctx, L, dev, n, d_src, d_off, d_slots, d_sizes, d_out, d_ooff, stride, st, stream, data, threads, check):
    """BASELINE.json configs[2] names levels 1 / 3 / 9: compress GB/s of the same 1 GiB, inputs in HBM, CPU arm beside it (level 5, the
    first of the lazy family, rides along)."""
    rec = {}
    for lvl in (1, 5, 9):
        def comp():
            check(L.zstdb200_compress_device(ctx.handle, lvl, n, d_src.data_ptr(), d_off.data_ptr(), d_slots.data_ptr(), stride, d_sizes.data_ptr(), st))
            check(L.zstdb200_compact_device(ctx.handle, n, d_slots.data_ptr(), stride, d_sizes.data_ptr(), d_out.data_ptr(), d_ooff.data_ptr(), st))
        ms = _time_ms(stream, comp, reps=2)
        ncpu = min(n, 1024 if lvl >= 9 else 2048 if lvl >= 5 else 4096)
        cpu = CpuRoundTrip(data[:ncpu], lvl, threads)
        tc, td, cs = cpu.run(); tc, td, cs = cpu.run()
        rec[f"L{lvl}"] = {"compress_gbs": n * CHUNK / (ms * 1e-3) / 1e9, "ms": ms, "cpu_compress_gbs": ncpu * CHUNK / tc / 1e9, "cpu_threads": threads, "cpu_sample_chunks": ncpu}
    return rec


def config3_record(args, ctx, L, dev, stream, st, check, threads):
    """BASELINE.json configs[3]: 10 000 frames made by the REFERENCE (chunk j mod 8192, levels cycling 1/3/9), decompress only,
    batch sizes 64 / 512 / 4096 / 10 000; frames resident in HBM.  The CPU arm decodes the same 10 000 frames."""
    import torch
    from zstd_jni_b200 import corpus
    Lr, kind = _cpu_lib()
    if kind != "reference":
        return {"unavailable": "oracle/_ref not built"}
    nf = 10000
    base = corpus.corpus(2048)                        # chunk j mod 2048 (bounded corpus build: 256 MiB), levels cycle 1/3/9
    bound = CHUNK + (CHUNK >> 8) + 64
    comp = np.zeros((nf, bound), dtype=np.uint8); sizes = np.zeros(nf, dtype=np.int64)
    def mk(idx):
        cctx = Lr.ZSTD_createCCtx(); cur = None
        for j in idx:
            lvl = (1, 3, 9)[j % 3]
            if lvl != cur: Lr.ZSTD_CCtx_setParameter(cctx, 100, lvl); cur = lvl
            sizes[j] = Lr.ZSTD_compress2(cctx, int(comp[j].ctypes.data), bound, int(base[j % 2048].ctypes.data), CHUNK)
        Lr.ZSTD_freeCCtx(cctx)
    with ThreadPoolExecutor(threads) as pool:
        list(pool.map(mk, [range(t, nf, threads) for t in range(threads)]))
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    packed = np.empty(int(offs[-1]), dtype=np.uint8)
    for j in range(nf): packed[offs[j]:offs[j + 1]] = comp[j, :sizes[j]]
    d_in = torch.from_numpy(packed).to(dev); d_ioff = torch.from_numpy(offs).to(dev)
    d_dst = torch.empty(nf * CHUNK, dtype=torch.uint8, device=dev); d_doff = torch.arange(0, (nf + 1) * CHUNK, CHUNK, dtype=torch.int64, device=dev)
    d_res = torch.zeros(nf, dtype=torch.int64, device=dev)
    rec = {"frames": nf, "compressed_bytes": int(offs[-1]), "made_by": "oracle/_ref ZSTD_compress2, levels 1/3/9 cycling", "batches": {}}
    for B in (64, 512, 4096, 10000):
        def dec():
            check(L.zstdb200_decompress_device(ctx.handle, B, d_in.data_ptr(), d_ioff.data_ptr(), d_dst.data_ptr(), d_doff.data_ptr(), d_res.data_ptr(), st))
        ms = _time_ms(stream, dec, reps=3)
        rec["batches"][str(B)] = {"ms": ms, "gbs_out": B * CHUNK / (ms * 1e-3) / 1e9, "hbm_gbs": (B * CHUNK + int(offs[B])) / (ms * 1e-3) / 1e9}
    expect = torch.from_numpy(base.reshape(-1)).to(dev)
    ok = bool((d_res == CHUNK).all()) and all(torch.equal(d_dst[j * CHUNK:(j + 1) * CHUNK], expect[(j % 2048) * CHUNK:(j % 2048 + 1) * CHUNK]) for j in range(0, nf, 97))
    rec["verified"] = ok
    back = np.empty((nf, CHUNK), dtype=np.uint8)
    def dd(idx):
        dctx = Lr.ZSTD_createDCtx()
        for j in idx: Lr.ZSTD_decompressDCtx(dctx, int(back[j].ctypes.data), CHUNK, int(comp[j].ctypes.data), int(sizes[j]))
        Lr.ZSTD_freeDCtx(dctx)
    with ThreadPoolExecutor(threads) as pool:
        parts = [range(t, nf, threads) for t in range(threads)]
        list(pool.map(dd, parts)); t0 = time.perf_counter(); list(pool.map(dd, parts)); tcpu = time.perf_counter() - t0
    rec["cpu_gbs_out"] = nf * CHUNK / tcpu / 1e9; rec["cpu_threads"] = threads
    return rec


def config4_record(args, data, threads):
    """BASELINE.json configs[4]: streaming through ZSTD_compressStream2 / ZSTD_decompressStream over direct buffers -- the Python
    mirrors of J/ZstdDirectBufferCompressingStreamNoFinalizer / ...DecompressingStreamNoFinalizer drive the C ABI exactly like the
    JNI glue (N/jni_directbuffercompress_zstd.c, N/jni_directbufferdecompress_zstd.c).  A 1 GiB slice of the 4 GiB stream (the
    corpus repeats every 1 GiB; the batch layer takes 1 GiB per call anyway); the CPU arm is the reference's streaming path on one
    thread -- a stream is a serial object in the reference -- over a bounded 128 MiB sample."""
    import torch
    from zstd_jni_b200.zstd import ByteBuffer, ZstdDirectBufferCompressingStream, ZstdDirectBufferDecompressingStream
    U = data.size
    src = ByteBuffer.allocateDirect(U); src.array[:] = data.reshape(-1)
    tgt = ByteBuffer.allocateDirect(U + (U >> 7) + 65536)
    back = ByteBuffer.allocateDirect(U)
    def once():
        src.clear(); tgt.clear(); back.clear()
        t0 = time.perf_counter()
        zc = ZstdDirectBufferCompressingStream(tgt, args.level); zc.compress(src); zc.close()
        t1 = time.perf_counter()
        tgt.flip()
        zd = ZstdDirectBufferDecompressingStream(tgt)
        while zd.hasRemaining():
            if zd.read(back) == 0 and not back.hasRemaining(): break
        zd.close()
        t2 = time.perf_counter()
        return t1 - t0, t2 - t1, tgt.limit()
    once(); tc, td, cs = once()
    ok = back.position() == U and bool((back.array[:U] == src.array[:U]).all())
    rec = {"bytes": U, "compressed_bytes": int(cs), "compress_gbs": U / tc / 1e9, "decompress_gbs": U / td / 1e9, "round_trip_gbs": U / (tc + td) / 1e9, "verified": ok,
           "api": "ZstdDirectBufferCompressingStream.compress / ZstdDirectBufferDecompressingStream.read over page-locked direct buffers (ZSTD_compressStream2 / ZSTD_decompressStream)"}
    Lr, kind = _cpu_lib()
    if kind == "reference":
        class _B(C.Structure): _fields_ = [("p", C.c_void_p), ("size", C.c_size_t), ("pos", C.c_size_t)]
        Lr.ZSTD_compressStream2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]; Lr.ZSTD_compressStream2.restype = C.c_size_t
        Lr.ZSTD_decompressStream.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]; Lr.ZSTD_decompressStream.restype = C.c_size_t
        ns = min(U, 128 << 20)
        sarr = np.ascontiguousarray(data.reshape(-1)[:ns]); out = np.empty(ns + (ns >> 7) + 65536, dtype=np.uint8); bk = np.empty(ns, dtype=np.uint8)
        cctx = Lr.ZSTD_createCCtx(); Lr.ZSTD_CCtx_setParameter(cctx, 100, args.level)
        ib = _B(int(sarr.ctypes.data), ns, 0); ob = _B(int(out.ctypes.data), out.size, 0)
        t0 = time.perf_counter()
        while True:
            r = Lr.ZSTD_compressStream2(cctx, C.byref(ob), C.byref(ib), 2)
            if r == 0: break
        t1 = time.perf_counter()
        Lr.ZSTD_freeCCtx(cctx)
        dctx = Lr.ZSTD_createDCtx()
        ib = _B(int(out.ctypes.data), ob.pos, 0); ob2 = _B(int(bk.ctypes.data), ns, 0)
        while ib.pos < ib.size:
            r = Lr.ZSTD_decompressStream(dctx, C.byref(ob2), C.byref(ib))
            if r > (1 << 63): break
        t2 = time.perf_counter()
        Lr.ZSTD_freeDCtx(dctx)
        rec["cpu"] = {"compress_gbs": ns / (t1 - t0) / 1e9, "decompress_gbs": ns / (t2 - t1) / 1e9, "round_trip_gbs": ns / (t2 - t0) / 1e9, "threads": 1,
                      "sample": f"first {ns >> 20} MiB through the reference's ZSTD_compressStream2 / ZSTD_decompressStream (one serial stream)", "verified": bool((bk == sarr).all())}
    return rec


def strong_scaling(args, ctx, L, dev, rank, world, local, check, barrier):
    """BASELINE.json configs[2] / SURVEY.md 8(e) items 1-3: ONE 1 GiB batch resident on GPU 0 -> NCCL scatter of contiguous chunk
    ranges -> every rank compresses its range -> all_gather of the frame sizes + exclusive scan -> gatherv of the packed frames
    into one contiguous stream on GPU 0; then the way back (scatter of the frames' byte ranges, decompress, gather of the chunks).
    Total work is fixed as N grows (strong scaling); times are CUDA events on every rank, max over ranks."""
    import torch
    import torch.distributed as dist
    from zstd_jni_b200 import corpus, sharding
    n_total = args.chunks
    stride = (L.ZSTD_compressBound(CHUNK) + 32 + 63) // 64 * 64
    s, e = sharding.shard_range(n_total, rank, world); cnt = e - s
    batch = torch.from_numpy(corpus.corpus(n_total).reshape(-1)).to(dev) if rank == 0 else None
    mine = torch.empty(max(cnt, 1) * CHUNK, dtype=torch.uint8, device=dev)
    d_off = torch.arange(0, (cnt + 1) * CHUNK, CHUNK, dtype=torch.int64, device=dev)
    d_slots = torch.empty(max(cnt, 1) * stride, dtype=torch.uint8, device=dev); d_sizes = torch.zeros(max(cnt, 1), dtype=torch.int64, device=dev)
    d_out = torch.empty(max(cnt, 1) * stride, dtype=torch.uint8, device=dev); d_ooff = torch.zeros(cnt + 1, dtype=torch.int64, device=dev)
    d_back = torch.empty(max(cnt, 1) * CHUNK, dtype=torch.uint8, device=dev); d_res = torch.zeros(max(cnt, 1), dtype=torch.int64, device=dev)
    stream_root = torch.empty(n_total * stride, dtype=torch.uint8, device=dev) if rank == 0 else None
    back_root = torch.empty(n_total * CHUNK, dtype=torch.uint8, device=dev) if rank == 0 else None
    cur = torch.cuda.Stream(device=dev); st = cur.cuda_stream        # an explicit stream: 0 would mean "the context's own stream" to the C ABI
    rec = {"total_bytes": n_total * CHUNK, "n_gpus": world, "levels": {}}
    torch.cuda.synchronize()
    with torch.cuda.stream(cur):
      for lvl in (1, 3, 9):
          def run(timed):
              ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
              ev[0].record(cur)
              sharding.scatter_chunks(batch, n_total, CHUNK, mine)
              ev[1].record(cur)
              check(L.zstdb200_compress_device(ctx.handle, lvl, cnt, mine.data_ptr(), d_off.data_ptr(), d_slots.data_ptr(), stride, d_sizes.data_ptr(), st))
              check(L.zstdb200_compact_device(ctx.handle, cnt, d_slots.data_ptr(), stride, d_sizes.data_ptr(), d_out.data_ptr(), d_ooff.data_ptr(), st))
              ev[2].record(cur)
              offs = sharding.global_offsets(sharding.gather_sizes(d_sizes[:cnt], n_total))
              ranges = sharding.rank_byte_ranges(offs, n_total, world)
              sharding.gatherv_bytes(d_out, ranges, stream_root)
              ev[3].record(cur)
              # way back: the root deals the frames' byte ranges out again, ranks decode, chunks come home
              lo, hi = ranges[rank]
              frames_local = torch.empty(max(hi - lo, 1), dtype=torch.uint8, device=dev)
              ops = []
              if rank == 0:
                  frames_local[: hi - lo].copy_(stream_root[lo:hi])
                  for r in range(1, world):
                      if ranges[r][1] > ranges[r][0]: ops.append(dist.P2POp(dist.isend, stream_root[ranges[r][0]:ranges[r][1]], r))
              elif hi > lo:
                  ops.append(dist.P2POp(dist.irecv, frames_local[: hi - lo], 0))
              if ops:
                  for w in dist.batch_isend_irecv(ops): w.wait()
              loc_off = (offs[s:e + 1] - offs[s]).contiguous()
              ev[4].record(cur)
              check(L.zstdb200_decompress_device(ctx.handle, cnt, frames_local.data_ptr(), loc_off.data_ptr(), d_back.data_ptr(), d_off.data_ptr(), d_res.data_ptr(), st))
              sharding.gather_fixed(d_back, n_total, CHUNK, back_root)
              ev[5].record(cur)
              torch.cuda.synchronize()
              t = [ev[k].elapsed_time(ev[k + 1]) for k in range(5)]
              return t, int(offs[-1])
          run(False); barrier()
          t, csize = run(True)
          tt = torch.tensor(t, dtype=torch.float64, device=dev)
          if world > 1: dist.all_reduce(tt, op=dist.ReduceOp.MAX)
          t = [float(x) for x in tt.tolist()]
          ok = True
          if rank == 0:
              ok = bool(torch.equal(back_root, batch))
          rec["levels"][f"L{lvl}"] = {"scatter_ms": t[0], "compress_ms": t[1], "sizes+gatherv_ms": t[2], "frames_scatter_ms": t[3], "decompress+gather_ms": t[4],
                                       "compress_path_ms": t[0] + t[1] + t[2], "round_trip_ms": sum(t), "compressed_bytes": csize,
                                       "compress_gbs": n_total * CHUNK / ((t[0] + t[1] + t[2]) * 1e-3) / 1e9, "round_trip_gbs": n_total * CHUNK / (sum(t) * 1e-3) / 1e9,
                                       "limiting": max((("scatter", t[0]), ("k_parse+k_entropy (per-frame tail)", t[1]), ("gatherv", t[2]), ("frames scatter", t[3]), ("decode+gather", t[4])), key=lambda kv: kv[1])[0],
                                       "verified": ok}
    rec["note"] = "strong scaling: efficiency(N) = round_trip_gbs(N) / (N x round_trip_gbs(1)) is computed by the reader from the per-N lines; N = 1 runs the same code without peers"
    return rec


if __name__ == "__main__":
    main()

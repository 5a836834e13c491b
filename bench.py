#!/usr/bin/env python3
"""bench.py -- BASELINE.json's metric on BASELINE.json's configs.

    python bench.py [--gpus N --steps K --warmup W] [--workload c1|c2|c3|c4|c5] [--impl reference]

Metric : GiB/s of INPUT (compress level 1 / Default, uncompress), next to the CPU baseline and the
         HBM roofline of the dominant kernel.  A "step" is one pass of the hot path over one batch.
Workloads (SURVEY.md 8d; all synthetic, seeded, generated on the device, larger than L2):
  c2 (default, the config BASELINE's metric is quoted on): 65536 x 64 KiB text blocks per GPU,
      compress level 1, one gzip member per block.  N>1: weak scaling, rank r takes blocks
      r*65536.., one NCCL all_gather of the member sizes (zippy_b200.sharding.gather_sizes).
  c1: zippy.compress(alice29.txt, dfGzip, BestSpeed) then uncompress: single-call latency (ms)
      through the drop-in calls, beside the oracle's (tests/bench.nim:28-64, README.md:41,63).
  c3: batch uncompress of 65536 gzip members = the reference's 23 .gz fixtures tiled, byte-exact.
  c4: compress level=Default of urls.10K x 6118 tiles (4 GiB), size vs the oracle's level -1.
  c5: mixed-entropy corpus, 131072 x 64 KiB blocks per GPU (8 GPUs = the 64 GiB of config 5), level 1;
      the sizes go through sharding.gather_sizes on NCCL and the e2e leg concatenates every rank's
      members at the gathered offsets into ONE host stream (a page-locked shared mapping).
The default line is c2's, with c1/c3/c4/c5 summaries under "extras" (N=1) or c5's (N>1), each with
its own roofline (live CUDA-event kernel times), cpu_baseline and e2e.

value  : whole-job GiB/s with inputs already resident in HBM (device variant of the C ABI).
e2e    : same metric through the host-buffer C-ABI call: pinned host input -> H2D -> kernels ->
         D2H of the result, all inside the timed region.  e2e_pageable: the same call on ordinary
         (not page-locked) memory.  pcie: plain cudaMemcpy H2D / D2H peaks measured in the same run.
--impl reference : the CPU path (oracle port of the reference; Nim is not available, so the
         reference itself cannot be built -- see DESIGN.md) on all host cores, bounded sample.
--dump-outputs DIR : after the timed steps, write what the selected workload's timed path returned in its
         last step as DIR/<name>.npy (see dump_members), so that two builds can be compared output for output.
"""
import argparse
import json
import mmap
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GIB = float(1 << 30)
BLOCK = 65536
BLOCKS_PER_GPU = 65536
C5_BLOCKS_PER_GPU = 131072
C3_MEMBERS = 65536
C4_TILES = 6118
DUMP_LIMIT = 64 * 10 ** 6   # bytes: every file --dump-outputs writes in one run, all ranks together
PUBLISHED_C1 = {"uncompress_alice29_ms": 0.233, "compress_best_speed_alice29_ms": 0.643,
                "hardware": "Ryzen 5 5600X, 1 thread (README.md:41,63); different machine"}


def sm64(x):
    x = (x + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    z = x
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return z ^ (z >> 31)


def text_corpus():
    from tests import util
    return util.text_corpus(util.load_corpus())


def bench_config(n, level, world):
    return {"workload": "C2: batch %d x 64 KiB synthetic text-entropy blocks per GPU, compress level=%d "
                        "dfGzip, one gzip member per block" % (n, level),
            "blocks_per_gpu": n, "block_bytes": BLOCK, "level": level, "data_format": "dfGzip",
            "l2": "inputs (4 GiB/GPU) larger than L2; no flush needed", "launch_group_chunks": n,
            "parallelism": "independent members sharded over %d GPU(s); NCCL all_gather of sizes" % world}


def block_offsets(T_len, first, count):
    return np.array([sm64(0xC2 + i) % (T_len - BLOCK) for i in range(first, first + count)], dtype=np.int64)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line).

    Primary source is NVML in-process (a few microseconds per query, so even a 0.3 s region gets
    dozens of samples); `nvidia-smi -lms` is the fallback when pynvml cannot open the device."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index):
        self.rows = []  # (sm_mhz, sm_max_mhz, set(reasons))
        self.stop = threading.Event()
        self.proc = None
        self.gpu = gpu_index
        self.nvml = None
        self.source = None

    def _open_nvml(self):
        import pynvml
        import torch
        pynvml.nvmlInit()
        h = None
        try:
            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except Exception:
                    idx = self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)  # probe
        self.nvml, self.h = pynvml, h
        self.masks = [(pynvml.nvmlClocksThrottleReasonHwSlowdown, "hw_slowdown"),
                      (pynvml.nvmlClocksThrottleReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                      (pynvml.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_thermal_slowdown"),
                      (pynvml.nvmlClocksThrottleReasonSwPowerCap, "sw_power_cap")]

    def _sample_nvml(self):
        n, h = self.nvml, self.h
        mx = float(n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM))
        while not self.stop.is_set():
            try:
                sm = float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
                bits = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.rows.append((sm, mx, {nm for m, nm in self.masks if bits & m}))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            self._open_nvml()
            self.source = "nvml"
            self.t = threading.Thread(target=self._sample_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.source = "nvidia-smi"
        self.t = threading.Thread(target=self._read_smi, daemon=True)
        self.t.start()

    def _read_smi(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) >= 7:
                try:
                    self.rows.append((float(f[0]), float(f[1]),
                                      {nm for nm, v in zip(self.NAMES, f[3:7]) if v.lower().startswith("active")}))
                except ValueError:
                    pass
            if self.stop.is_set():
                break

    def mark(self):
        """Samples taken before this point (start-up, idle clocks) are dropped."""
        self.first = len(self.rows)

    def snapshot(self):
        """Summary of the samples since mark(); the sampler keeps running."""
        if self.source is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["no clock source (nvml, nvidia-smi)"]}
        rows = self.rows[getattr(self, "first", 0):]
        sm = [r[0] for r in rows]
        reasons = set()
        for r in rows:
            reasons |= r[2]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(r[1] for r in rows) if rows else None,
                "samples": len(sm), "source": self.source, "reasons": sorted(reasons)}

    def finish(self):
        out = self.snapshot()
        self.stop.set()
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        return out


def host_threads():
    """Threads the CPU arm may really use: the affinity mask, capped by a cgroup CPU quota if there is one."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(int(q) / float(p) + 0.5)))
    except Exception:
        pass
    return max(1, n)


# ======================================================================================
# CPU legs (the oracle port of the reference, and system zlib as README's own comparator)
# ======================================================================================
def _c2_sample(T, nb):
    offs = block_offsets(len(T), 0, min(nb, 4096))
    Tn = np.frombuffer(T, dtype=np.uint8)
    buf = np.empty(nb * BLOCK, dtype=np.uint8)
    for i in range(nb):
        s = int(offs[i % len(offs)])
        buf[i * BLOCK:(i + 1) * BLOCK] = Tn[s:s + BLOCK]
    return buf, np.arange(nb + 1, dtype=np.uint64) * BLOCK


def cpu_compress_leg(make, unit_bytes, level, seconds, threads, label, max_units=65536):
    """Oracle compress of independent inputs on `threads` host threads, sized to run ~`seconds`.
    make(k) -> (uint8 buffer, offsets) of k inputs of unit_bytes each."""
    from oracle import oracle as o
    pilot = max(threads * 2, 4)
    buf, bo = make(pilot)
    t0 = time.perf_counter()
    o.compress_batch(buf, bo, level, o.dfGzip, threads=threads)
    dt = max(time.perf_counter() - t0, 1e-3)
    k = int(min(max(pilot, pilot * seconds / dt), max_units))
    buf, bo = make(k)
    t0 = time.perf_counter()
    total, lens, st = o.compress_batch(buf, bo, level, o.dfGzip, threads=threads)
    dt = time.perf_counter() - t0
    assert not st.any()
    nbytes = int(bo[-1])
    return {"value": nbytes / GIB / dt, "unit": "GiB/s", "cores": threads, "kind": "port",
            "sample": "%d x %s, oracle level %d gzip, %d threads, %.1f s" % (k, label, level, threads, dt),
            "ratio": float(total) / nbytes}, k, dt


def cpu_baseline(T, n_blocks_hint, seconds=12.0, threads=None, level=1):
    """Oracle (port of the reference's level-1 path) over independent C2 blocks on all host cores."""
    cores = threads or host_threads()
    return cpu_compress_leg(lambda k: _c2_sample(T, k), BLOCK, level, seconds, cores, "64 KiB C2 text blocks")


def zlib_compress_leg(buf, offsets, level, threads, seconds=2.0):
    """System zlib (README's comparator, tests/bench.nim:30-46) over the same inputs; zlib releases the GIL."""
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    mv = memoryview(buf)
    items = [(int(offsets[i]), int(offsets[i + 1])) for i in range(len(offsets) - 1)]

    def one(ab):
        c = zlib.compressobj(level, zlib.DEFLATED, 31)
        return len(c.compress(mv[ab[0]:ab[1]])) + len(c.flush())

    t0 = time.perf_counter()
    done, out = 0, 0
    with ThreadPoolExecutor(threads) as ex:
        while time.perf_counter() - t0 < seconds or done == 0:
            out = sum(ex.map(one, items))
            done += 1
    dt = time.perf_counter() - t0
    nbytes = int(offsets[-1]) * done
    return {"value": nbytes / GIB / dt, "unit": "GiB/s", "cores": threads, "kind": "zlib-%s" % zlib.ZLIB_RUNTIME_VERSION,
            "level": level, "ratio": out / float(int(offsets[-1]))}


def cpu_uncompress_leg(members, out_bytes, seconds, threads):
    """Oracle inflate (port of inflate.nim) of the given gzip members on `threads` host threads."""
    from oracle import oracle as o
    # enough members that every thread has many (and the few large fixtures do not decide the balance)
    reps = max(1, (threads * 8 + len(members) - 1) // len(members), int((threads * (24 << 20)) // max(out_bytes, 1)))
    lens = np.array([len(m) for m in members] * reps, dtype=np.uint64)
    base = np.frombuffer(b"".join(members) * reps, dtype=np.uint8)
    mo = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=mo[1:])
    t0 = time.perf_counter()
    total, _, st = o.uncompress_batch(base, mo, o.dfGzip, threads=threads)
    dt = max(time.perf_counter() - t0, 1e-4)
    rounds = int(max(1, min(64, seconds / dt)))
    t0 = time.perf_counter()
    for _ in range(rounds):
        total, _, st = o.uncompress_batch(base, mo, o.dfGzip, threads=threads)
    dt = time.perf_counter() - t0
    assert not st.any() and int(total) == out_bytes * reps
    return {"out_gibs": rounds * int(total) / GIB / dt, "in_gibs": rounds * int(mo[-1]) / GIB / dt, "cores": threads,
            "kind": "port", "sample": "%d gzip members x %d rounds, oracle inflate, %d threads, %.1f s"
            % (len(lens), rounds, threads, dt)}


def zlib_uncompress_leg(members, threads, seconds=1.5):
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    t0 = time.perf_counter()
    done, out = 0, 0
    with ThreadPoolExecutor(threads) as ex:
        while time.perf_counter() - t0 < seconds or done == 0:
            out = sum(ex.map(lambda m: len(zlib.decompress(m, 47)), members))
            done += 1
    dt = time.perf_counter() - t0
    return {"out_gibs": done * out / GIB / dt, "cores": threads, "kind": "zlib-%s" % zlib.ZLIB_RUNTIME_VERSION}


def cpu_uncompress_baseline(T, seconds=4.0, threads=None):
    """Oracle inflate of level-1 gzip members of C2 blocks, all host cores."""
    from oracle import oracle as o
    cores = threads or host_threads()
    offs = block_offsets(len(T), 0, 512)
    members = [o.compress(T[int(s):int(s) + BLOCK], 1, o.dfGzip) for s in offs]
    return cpu_uncompress_leg(members, len(members) * BLOCK, seconds, cores)


def cpu_checksum_legs(seconds=0.5):
    """crc32 / adler32 of a 64 MiB buffer, one thread: the oracle's SIMD forms (what the reference runs on
    amd64: PCLMUL / SSSE3) and system zlib."""
    import zlib
    from oracle import oracle as o
    b = np.random.default_rng(1).integers(0, 256, 64 << 20, dtype=np.uint8).tobytes()
    out = {}
    for name, f in (("oracle_crc32", o.crc32), ("oracle_adler32", o.adler32), ("zlib_crc32", zlib.crc32),
                    ("zlib_adler32", zlib.adler32)):
        f(b)
        t0 = time.perf_counter()
        k = 0
        while time.perf_counter() - t0 < seconds:
            f(b)
            k += 1
        out[name + "_gbs"] = k * len(b) / (time.perf_counter() - t0) / 1e9
    out["cores"] = 1
    return out


# ======================================================================================
# GPU side
# ======================================================================================
class Env:
    pass


def make_env(args):
    import torch
    import torch.distributed as dist
    import zippy_b200 as z
    from zippy_b200 import sharding
    e = Env()
    e.rank = int(os.environ.get("RANK", "0"))
    e.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    e.world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(e.local_rank)
    # before any page-locked buffer exists: run on (and first-touch memory of) the GPU's NUMA node
    e.numa = sharding.bind_to_gpu_numa_node(e.local_rank) if not args.no_numa else {"bound": False, "off": True}
    e.dev = torch.device("cuda", e.local_rank)
    if e.world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=e.dev)
    e.torch, e.dist, e.z, e.sharding = torch, dist, z, sharding
    e.ctx = z.Context(e.local_rank)
    e.stream = torch.cuda.current_stream()
    e.ctx.set_stream(e.stream.cuda_stream or e.ctx.LEGACY_DEFAULT_STREAM)   # same stream as torch's work: ordered
    e.ev0 = torch.cuda.Event(enable_timing=True)
    e.ev1 = torch.cuda.Event(enable_timing=True)
    try:
        e.peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        e.peaks = {}
    e.hbm_peak = float(e.peaks.get("hbm_gbs", 6650.0))
    e.peak_source = "measured" if "hbm_gbs" in e.peaks else "fallback"
    try:
        e.traffic = json.load(open(os.path.join(ROOT, "profiles", "latest_traffic.json")))
    except Exception:
        e.traffic = {}
    return e


def sync_all(e):
    e.torch.cuda.synchronize()
    if e.world > 1:
        e.dist.barrier()
        e.torch.cuda.synchronize()


def timed(e, fn, steps):
    """K calls of fn bracketed by barrier + synchronize, CUDA events on the launching stream, max over ranks.
    SM clocks / throttle reasons are sampled during exactly this region (e.last_clocks)."""
    sync_all(e)
    e.clocks.mark()
    e.ev0.record(e.stream)
    for _ in range(steps):
        fn()
    e.ev1.record(e.stream)
    sync_all(e)
    e.last_clocks = e.clocks.snapshot()
    t = e.torch.tensor([e.ev0.elapsed_time(e.ev1)], dtype=e.torch.float64, device=e.dev)
    if e.world > 1:
        e.dist.all_reduce(t, op=e.dist.ReduceOp.MAX)
    return float(t.item()) / steps


def roofline(e, kernel, kernel_ms, algo_bytes, all_ms=None):
    achieved = algo_bytes / (kernel_ms / 1e3) / 1e9 if kernel_ms > 0 else 0.0
    tr = e.traffic.get(kernel)
    r = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": e.hbm_peak, "unit": "GB/s",
         "frac": achieved / e.hbm_peak, "peak_source": e.peak_source, "algorithmic_bytes_per_launch": int(algo_bytes),
         "kernel_ms": kernel_ms, "traffic": tr.get("dram_bytes_per_launch") if isinstance(tr, dict) else tr}
    if isinstance(tr, dict):
        r["traffic_source"] = tr.get("source")
    if all_ms is not None:
        r["kernel_ms_all"] = all_ms
    return r


def pinned(e, nbytes):
    return e.torch.empty(int(nbytes), dtype=e.torch.uint8).pin_memory()


def pcie_peaks(e, nbytes=1 << 30):
    """Plain cudaMemcpyAsync of page-locked memory, best of 3, in the same run: what 'PCIe-bound' means here."""
    t = e.torch
    h = pinned(e, nbytes)
    d = t.empty(nbytes, dtype=t.uint8, device=e.dev)
    out = {}
    for name, (dst, src) in (("h2d_gbs", (d, h)), ("d2h_gbs", (h, d))):
        best = 1e9
        for _ in range(4):
            t.cuda.synchronize()
            e.ev0.record(e.stream)
            dst.copy_(src, non_blocking=True)
            e.ev1.record(e.stream)
            t.cuda.synchronize()
            best = min(best, e.ev0.elapsed_time(e.ev1))
        out[name] = nbytes / (best / 1e3) / 1e9
    # both directions at once (two streams), best of 3: what a pipelined host call can hope for
    s2 = t.cuda.Stream()
    h2 = pinned(e, nbytes)
    d2 = t.empty(nbytes, dtype=t.uint8, device=e.dev)
    best = 1e9
    for _ in range(4):
        t.cuda.synchronize()
        t0 = time.perf_counter()
        d.copy_(h, non_blocking=True)
        with t.cuda.stream(s2):
            h2.copy_(d2, non_blocking=True)
        t.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    out["duplex_each_gbs"] = nbytes / best / 1e9
    out["bytes"] = nbytes
    return out


def gen_c2(e, n, first):
    t = e.torch
    T = text_corpus()
    T_d = t.frombuffer(bytearray(T), dtype=t.uint8).to(e.dev)
    offs = t.from_numpy(block_offsets(len(T), first, n)).to(e.dev)
    windows = T_d.unfold(0, BLOCK, 1)
    d_src = t.empty(n * BLOCK, dtype=t.uint8, device=e.dev)
    for s in range(0, n, 4096):
        k = min(n, s + 4096)
        d_src[s * BLOCK:k * BLOCK] = t.index_select(windows, 0, offs[s:k]).reshape(-1)
    t.cuda.synchronize()   # the ctx runs on its own stream: inputs are complete before the first call
    return d_src, T


def gen_c5(e, nb, first):
    """SURVEY 8d config 5: class = sm64(0xC5 + i) mod 8: 0-3 text, 4 urls.10K window, 5 html window,
    6 random bytes, 7 run-length blob (tests/stress.nim:13-24)."""
    from tests import util
    t = e.torch
    corpus = util.load_corpus()
    T = util.text_corpus(corpus)
    cls = np.array([sm64(0xC5 + first + i) % 8 for i in range(nb)], dtype=np.int64)
    d_src = t.empty(nb * BLOCK, dtype=t.uint8, device=e.dev)
    view = d_src.view(nb, BLOCK)
    for name, sel in (("text", cls < 4), ("urls", cls == 4), ("html", cls == 5)):
        raw = T if name == "text" else corpus["urls.10K" if name == "urls" else "html"]
        idx = np.nonzero(sel)[0]
        if not len(idx):
            continue
        offs_b = np.array([(sm64(0xC5C5 + first + int(i)) >> 3) % (len(raw) - BLOCK) for i in idx], dtype=np.int64)
        win = t.frombuffer(bytearray(raw), dtype=t.uint8).to(e.dev).unfold(0, BLOCK, 1)
        for s0 in range(0, len(idx), 4096):
            rows = t.index_select(win, 0, t.from_numpy(offs_b[s0:s0 + 4096]).to(e.dev))
            view[t.from_numpy(idx[s0:s0 + 4096]).to(e.dev)] = rows
    g = t.Generator(device=e.dev)
    g.manual_seed(0xC5 + first)
    idx = t.from_numpy(np.nonzero(cls == 6)[0]).to(e.dev)
    if len(idx):
        view[idx] = t.randint(0, 256, (len(idx), BLOCK), dtype=t.uint8, device=e.dev, generator=g)
    idx = t.from_numpy(np.nonzero(cls == 7)[0]).to(e.dev)
    if len(idx):
        need = len(idx) * BLOCK
        runs = t.randint(1, 256, (need // 100 + 1024,), device=e.dev, generator=g)
        vals = t.randint(0, 256, (len(runs),), dtype=t.uint8, device=e.dev, generator=g)
        blob = t.repeat_interleave(vals, runs)[:need]
        assert blob.numel() == need
        view[idx] = blob.view(len(idx), BLOCK)
    t.cuda.synchronize()
    return d_src, cls


def check_members(e, d_src, src_offs, d_dst, oo, idxs):
    """The oracle AND zlib inflate these members of the GPU's output back to the input."""
    import zlib
    from oracle import oracle as o
    for i in idxs:
        m = d_dst[int(oo[i]):int(oo[i + 1])].cpu().numpy().tobytes()
        want = d_src[int(src_offs[i]):int(src_offs[i + 1])].cpu().numpy().tobytes()
        assert o.uncompress(m) == want and zlib.decompress(m, 31) == want, "parity failure on member %d" % i


def measure_compress(e, d_src, src_offs, level, steps, warmup, n_total_members, first_member, do_e2e=True,
                     e2e_steps=None, pageable=False, concat=False, parity_idx=range(8), roundtrip=True):
    """Device-resident compress of this rank's members (+ NCCL size exchange when world > 1), the
    host-buffer e2e, and the live roofline of the dominant kernel."""
    t, z, ctx = e.torch, e.z, e.ctx
    n = len(src_offs) - 1
    in_bytes = int(src_offs[n])
    cap = in_bytes + 96 * n + 4096
    cap += (-cap) % 4
    d_dst = t.empty(cap, dtype=t.uint8, device=e.dev)
    state = {}

    def step_device():
        oo = ctx.compress_batch_device(d_src.data_ptr(), src_offs, level, z.dfGzip, d_dst.data_ptr(), cap)
        if e.world > 1:   # the path's one exchange: every rank learns every member's compressed size
            sizes, goffs = e.sharding.gather_sizes((oo[1:] - oo[:-1]).astype(np.int64), n_total_members, device=e.dev,
                                                   on_device=True)   # global concatenation offsets, left on the device
            state["goffs"] = goffs
        state["oo"] = oo

    for _ in range(max(warmup, 1)):
        step_device()
    sync_all(e)
    oo = state["oo"]
    comp_bytes = int(oo[n])
    res = {"comp_bytes": comp_bytes, "in_bytes": in_bytes, "ratio": comp_bytes / float(in_bytes)}
    if e.rank == 0:
        check_members(e, d_src, src_offs, d_dst, oo, parity_idx)
    if roundtrip:   # the GPU inflates the whole batch back: bit-exact at full size
        d_back = t.empty(in_bytes, dtype=t.uint8, device=e.dev)
        lens, st = ctx.uncompress_batch_device(d_dst.data_ptr(), oo, z.dfDetect, d_back.data_ptr(), src_offs)
        ti = ctx.timing()
        assert not st.any() and bool((lens == (src_offs[1:] - src_offs[:-1])).all()), "GPU inflate reported errors"
        assert t.equal(d_back, d_src), "round trip mismatch at full size"
        del d_back
        res["roundtrip_inflate_ms"] = ti["inflate_ms"] + ti["verify_ms"]
        res["roundtrip_inflate_only_ms"] = ti["inflate_ms"]

    kern = {"lz_ms": 0.0, "huff_ms": 0.0, "scan_ms": 0.0, "pack_ms": 0.0}
    launches = [0]

    def step_timed():
        step_device()
        tm = ctx.timing()
        for k in kern:
            kern[k] += tm[k]
        launches[0] += tm["kernel_launches"]

    ms = timed(e, step_timed, steps)
    if e.dump_dir:   # here, before the e2e legs: c5's writes d_dst again through the host-input call
        from zippy_b200 import _native
        sizes, inv = np.unique(np.diff(src_offs), return_inverse=True)
        bound = np.array([_native.lib().zb200_compress_bound(int(s), z.dfGzip) for s in sizes], dtype=np.uint64)
        dump_members(e, d_dst, state["oo"], bound[inv])
    res["clocks"] = e.last_clocks
    res["ms_per_step"] = ms
    res["value"] = e.world * in_bytes / GIB / (ms / 1e3)   # weak scaling: every rank has in_bytes
    res["gpu_launches"] = int(launches[0])
    per = {k: v / steps for k, v in kern.items()}
    dom = max(per, key=per.get)
    res["roofline"] = roofline(e, "k_lz2" if (dom == "lz_ms" and (level == -1 or level >= 2)) else "k_" + dom[:-3],
                               per[dom], in_bytes + comp_bytes, per)

    if do_e2e:
        from zippy_b200 import _native
        L = _native.lib()
        ks = e2e_steps or steps
        h_src = pinned(e, in_bytes)
        h_src.copy_(d_src)
        out_offs = np.zeros(n + 1, dtype=np.uint64)
        stat = np.zeros(n, dtype=np.int32)
        if not concat:
            hcap = comp_bytes + (64 << 20)
            h_dst = pinned(e, hcap)

            def step_host():
                rc = L.zb200_compress_batch(ctx._h, h_src.data_ptr(), src_offs.ctypes.data, n, level, z.dfGzip,
                                            None, h_dst.data_ptr(), hcap, out_offs.ctypes.data, stat.ctypes.data)
                assert rc == 0, rc
                if e.world > 1:
                    e.sharding.gather_sizes((out_offs[1:] - out_offs[:-1]).astype(np.int64), n_total_members, device=e.dev,
                                            on_device=True)

            for _ in range(2):
                step_host()
            ms2 = timed(e, step_host, ks)
            th = ctx.timing()
            assert int(out_offs[n]) == comp_bytes
            res["e2e"] = {"value": e.world * in_bytes / GIB / (ms2 / 1e3), "unit": "GiB/s", "ms_per_step": ms2,
                          "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": comp_bytes,
                          "h2d_ms": th["h2d_ms"], "d2h_ms": th["d2h_ms"], "host_memory": "page-locked"}
            if pageable:
                # the same call on ordinary memory (what a Nim string is): staged through the library's pinned ring
                p_src = np.empty(in_bytes, dtype=np.uint8)
                p_src[:] = h_src.numpy()
                p_dst = np.empty(hcap, dtype=np.uint8)

                def step_pageable():
                    rc = L.zb200_compress_batch(ctx._h, p_src.ctypes.data, src_offs.ctypes.data, n, level, z.dfGzip,
                                                None, p_dst.ctypes.data, hcap, out_offs.ctypes.data, stat.ctypes.data)
                    assert rc == 0, rc

                step_pageable()
                ms3 = timed(e, step_pageable, max(1, ks // 2))
                assert int(out_offs[n]) == comp_bytes and bytes(p_dst[:4096]) == bytes(h_dst[:4096].numpy())
                res["e2e_pageable"] = {"value": e.world * in_bytes / GIB / (ms3 / 1e3), "unit": "GiB/s", "ms_per_step": ms3,
                                       "host_memory": "pageable (numpy)"}
                del p_src, p_dst
            res["_h_dst"] = h_dst
            res["_out_offs"] = out_offs.copy()
        else:
            # config 5: every rank's members land at the gathered offsets of ONE host stream
            res["e2e"] = e2e_concat(e, L, h_src, d_dst, cap, src_offs, level, n_total_members, first_member, ks, comp_bytes)
        del h_src
    res["_d_dst"] = d_dst
    res["_oo"] = oo
    return res


def e2e_concat(e, L, h_src, d_dst, cap, src_offs, level, n_total, first_member, steps, comp_bytes):
    """H2D + kernels (members stay on the device) -> NCCL all_gather of the sizes -> each rank copies its
    shard to its global offset in one shared, page-locked host mapping: the concatenated stream."""
    z, ctx = e.z, e.ctx
    n = len(src_offs) - 1
    path = "/dev/shm/zb200_concat_%s.bin" % os.environ.get("MASTER_PORT", str(os.getpid()))
    out_offs = [None]
    goffs_box = [None]
    mapping = {}

    def ensure_mapping(total):
        if "arr" in mapping:
            return
        lo, hi = int(goffs_box[0][first_member]), int(goffs_box[0][first_member + n])
        # one mapping shared by every rank (tmpfs); when /dev/shm is too small for the stream, each rank keeps
        # its slice in private page-locked memory instead (same offsets, no shared view)
        try:
            sv = os.statvfs("/dev/shm")
            fits = sv.f_bavail * sv.f_frsize > total + (256 << 20)
        except OSError:
            fits = False
        flag = e.torch.tensor([1 if fits else 0], device=e.dev)
        if e.world > 1:
            e.dist.all_reduce(flag, op=e.dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            buf = pinned(e, hi - lo + 64)
            mapping.update(arr=buf.numpy(), base=lo, keep=buf, kind="per-rank page-locked slices (/dev/shm too small for one mapping)")
            return
        if e.rank == 0:
            with open(path, "wb") as f:
                f.truncate(total)
        if e.world > 1:
            e.dist.barrier()
        f = open(path, "r+b")
        mm = mmap.mmap(f.fileno(), total)
        arr = np.frombuffer(mm, dtype=np.uint8)
        a0, a1 = lo & ~4095, min(total, (hi + 4095) & ~4095)
        arr[a0:a1:4096] = 0                       # touch the pages (on this rank's NUMA node)
        kind = "one shared host mapping, this rank's slice page-locked"
        try:
            e.z.host_register(arr.ctypes.data + a0, a1 - a0)
            mapping["reg"] = (a0, a1)
        except Exception:
            kind = "one shared host mapping (cudaHostRegister refused it: pageable copies)"
        mapping.update(mm=mm, arr=arr, f=f, base=0, kind=kind)

    def step():
        oo = ctx.compress_batch_h2d(h_src.data_ptr(), src_offs, level, z.dfGzip, d_dst.data_ptr(), cap)
        sizes, goffs = e.sharding.gather_sizes((oo[1:] - oo[:-1]).astype(np.int64), n_total, device=e.dev)
        out_offs[0], goffs_box[0] = oo, goffs
        ensure_mapping(int(goffs[-1]))
        ctx.download(d_dst.data_ptr(), mapping["arr"].ctypes.data + int(goffs[first_member]) - mapping["base"], int(oo[n]))

    for _ in range(2):
        step()
    ms = timed(e, step, steps)
    goffs = goffs_box[0]
    assert int(out_offs[0][n]) == comp_bytes
    # parity on the concatenated stream: rank 0 inflates members from every shard it can see with the oracle
    ok = True
    total = int(goffs[-1])
    shared = "mm" in mapping
    if e.rank == 0:
        from oracle import oracle as o
        arr = mapping["arr"]
        for r in range(e.world if shared else 1):
            lo, _ = e.sharding.shard_range(n_total, r, e.world)
            for k in (0, 1, n - 1):
                a, b = int(goffs[lo + k]) - mapping["base"], int(goffs[lo + k + 1]) - mapping["base"]
                ok = ok and len(o.uncompress(bytes(arr[a:b]))) == BLOCK
        if shared:
            assert len(arr) == total
    sync_all(e)
    if "reg" in mapping:
        e.z.host_unregister(mapping["arr"].ctypes.data + mapping["reg"][0])
    kind = mapping["kind"]
    mapping.pop("arr")
    if shared:
        try:
            mapping["mm"].close()
        except BufferError:
            pass
        mapping["f"].close()
        if e.world > 1:
            e.dist.barrier()
        if e.rank == 0:
            try:
                os.unlink(path)
            except OSError:
                pass
    return {"value": e.world * int(src_offs[n]) / GIB / (ms / 1e3), "unit": "GiB/s", "ms_per_step": ms,
            "h2d_bytes_per_step": int(src_offs[n]), "d2h_bytes_per_step": comp_bytes,
            "host_memory": "input page-locked; output = one concatenated stream of %d bytes: %s" % (total, kind),
            "concat_parity": "oracle inflated 3 members of every rank's shard from the concatenated stream: %s" % ok}


def measure_uncompress(e, d_comp, comp_offs, out_sizes, steps, warmup, do_e2e=True, h_comp=None):
    """Device-resident batch uncompress (inflate + trailer verification) and the host-buffer e2e."""
    t, z, ctx = e.torch, e.z, e.ctx
    n = len(comp_offs) - 1
    doffs = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(out_sizes, out=doffs[1:])
    out_bytes, in_bytes = int(doffs[n]), int(comp_offs[n] - comp_offs[0])
    d_out = t.empty(out_bytes + 64, dtype=t.uint8, device=e.dev)
    acc = {"inflate_ms": 0.0, "verify_ms": 0.0, "launches": 0}

    def step():
        lens, st = ctx.uncompress_batch_device(d_comp.data_ptr(), comp_offs, z.dfDetect, d_out.data_ptr(), doffs)
        tm = ctx.timing()
        acc["inflate_ms"] += tm["inflate_ms"]
        acc["verify_ms"] += tm["verify_ms"]
        acc["launches"] += tm["kernel_launches"]
        acc["last"] = (lens, st)
        return lens, st

    for _ in range(max(1, warmup)):
        lens, st = step()
    assert not st.any() and bool((lens == out_sizes).all())
    acc.update(inflate_ms=0.0, verify_ms=0.0, launches=0)
    ms = timed(e, step, steps)
    per = {"inflate_ms": acc["inflate_ms"] / steps, "verify_ms": acc["verify_ms"] / steps}
    res = {"clocks": e.last_clocks, "ms_per_step": ms, "in_bytes": in_bytes, "out_bytes": out_bytes, "in_gibs": in_bytes / GIB / (ms / 1e3),
           "out_gibs": out_bytes / GIB / (ms / 1e3), "gpu_launches": acc["launches"],
           "roofline": roofline(e, "k_inflate", per["inflate_ms"], in_bytes + out_bytes, per), "_d_out": d_out, "_doffs": doffs,
           "_lens": acc["last"][0], "_st": acc["last"][1]}
    if do_e2e:
        from zippy_b200 import _native
        L = _native.lib()
        if h_comp is None:
            h_comp = pinned(e, in_bytes)
            h_comp.copy_(d_comp[int(comp_offs[0]):int(comp_offs[n])])
        h_out = pinned(e, out_bytes + 64)
        lens_b = np.zeros(n, dtype=np.uint64)
        stat = np.zeros(n, dtype=np.int32)
        co = (comp_offs - comp_offs[0]).astype(np.uint64)

        def step_back():
            rc = L.zb200_uncompress_batch(ctx._h, h_comp.data_ptr(), co.ctypes.data, n, z.dfDetect, h_out.data_ptr(),
                                          doffs.ctypes.data, lens_b.ctypes.data, stat.ctypes.data)
            assert rc == 0, rc

        step_back()
        sync_all(e)
        assert not stat.any() and bool((lens_b == out_sizes).all())
        chk = min(out_bytes, 64 << 20)
        assert t.equal(h_out[:chk], d_out[:chk].cpu()), "host uncompress differs from the device-resident result"
        ms3 = timed(e, step_back, steps)
        tb = ctx.timing()
        res["e2e"] = {"value": in_bytes / GIB / (ms3 / 1e3), "unit": "GiB/s", "out_gibs": out_bytes / GIB / (ms3 / 1e3),
                      "in_gibs": in_bytes / GIB / (ms3 / 1e3), "ms_per_step": ms3, "h2d_bytes_per_step": in_bytes,
                      "d2h_bytes_per_step": out_bytes, "h2d_ms": tb["h2d_ms"], "d2h_ms": tb["d2h_ms"],
                      "inflate_ms": tb["inflate_ms"] + tb["verify_ms"], "host_memory": "page-locked"}
        # the same bytes as ONE plain device -> host copy into the same buffer: the floor of the copy-out leg
        t.cuda.synchronize()
        e.ev0.record(e.stream)
        h_out[:out_bytes].copy_(d_out[:out_bytes], non_blocking=True)
        e.ev1.record(e.stream)
        t.cuda.synchronize()
        res["e2e"]["d2h_plain_gbs"] = out_bytes / (e.ev0.elapsed_time(e.ev1) / 1e3) / 1e9
        del h_out
    return res


def run_checksums(e, args):
    """Standalone crc32 / adler32 (SURVEY 8 rows A9 / A10): 65 536 x 64 KiB buffers and the same 4 GiB as ONE
    buffer, device-resident, kernel times from the library's own CUDA events; values checked against zlib."""
    import zlib
    t, ctx = e.torch, e.ctx
    n = args.blocks
    g = t.Generator(device=e.dev)
    g.manual_seed(1)
    d_src = t.randint(0, 256, (n * BLOCK,), dtype=t.uint8, device=e.dev, generator=g)
    t.cuda.synchronize()
    head = d_src[:BLOCK].cpu().numpy().tobytes()
    whole = d_src[:64 << 20].cpu().numpy().tobytes() if n * BLOCK >= (64 << 20) else None
    out = {"workload": "crc32 / adler32 of %d x 64 KiB buffers and of one %d MiB buffer, device-resident" % (n, n // 16),
           "cpu_1_thread": cpu_checksum_legs() if not args.no_cpu else None}
    for label, offs in (("batch", np.arange(n + 1, dtype=np.uint64) * BLOCK), ("one_buffer", np.array([0, n * BLOCK], dtype=np.uint64))):
        for kind in ("crc32", "adler32"):
            times = []
            for _ in range(6):   # the first calls also pay for the piece table upload and cold TLBs
                vals = ctx.checksum_batch_device(d_src.data_ptr(), offs, kind)
                times.append(ctx.timing()["checksum_ms"])
            ms = float(np.median(times[2:]))
            if label == "batch":
                assert int(vals[0]) == (zlib.crc32(head) if kind == "crc32" else zlib.adler32(head))
            elif whole is not None and n * BLOCK == (64 << 20):
                assert int(vals[0]) == (zlib.crc32(whole) if kind == "crc32" else zlib.adler32(whole))
            gbs = n * BLOCK / (ms / 1e3) / 1e9
            out["%s_%s" % (kind, label)] = {"ms": ms, "GB_s": gbs, "roofline": {
                "bound": "hbm", "kernel": "k_piece_checksum (+ fold / combine)", "achieved": gbs, "peak": e.hbm_peak, "unit": "GB/s",
                "frac": gbs / e.hbm_peak, "peak_source": e.peak_source, "algorithmic_bytes_per_launch": n * BLOCK, "kernel_ms": ms,
                "traffic": None}}
    del d_src
    return out


def strip(d):
    return {k: v for k, v in d.items() if not k.startswith("_")}


def save_output(e, name, arr):
    """DIR/<name>.npy (rank<r>_<name>.npy when several ranks each hold a shard)."""
    os.makedirs(e.dump_dir, exist_ok=True)
    prefix = "rank%d_" % e.rank if e.world > 1 else ""
    np.save(os.path.join(e.dump_dir, prefix + name + ".npy"), arr)


def dump_members(e, d_buf, offsets, max_bytes, **returned):
    """--dump-outputs for a batch call: member i of the result lies in d_buf[offsets[i]:offsets[i + 1]].
    Every member is covered by offsets.npy, crc32.npy and the call's other per-member results (`returned`),
    all float64, which holds them exactly.  The CRC-32s come from the build's own checksum kernel: a
    fingerprint of the bytes, not an independent check of them.  sample_bytes.npy holds the bytes (as
    float32) of the whole members listed in sample_index.npy, concatenated in that order.  The sample is a
    seeded draw over max_bytes, a bound of each member's size known before the call, so it does not depend
    on what the build produced; it is sized so that the files of all ranks together stay within DUMP_LIMIT."""
    n = len(offsets) - 1
    crc = e.ctx.checksum_batch_device(d_buf.data_ptr(), offsets, "crc32")
    full = dict(offsets=offsets, crc32=crc, **returned)
    budget = DUMP_LIMIT // e.world - sum(8 * len(a) + 256 for a in full.values()) - 2 * 256   # 256: .npy header
    assert budget >= 0, "too many members per rank for a %d-byte dump" % DUMP_LIMIT
    order = np.random.default_rng(0).permutation(n)
    cost = 4 * max_bytes[order].astype(np.int64) + 8   # float32 bytes + a float64 index
    idx = np.sort(order[:np.searchsorted(np.cumsum(cost), budget, side="right")])
    sample = e.torch.cat([d_buf[int(offsets[i]):int(offsets[i + 1])] for i in idx]) if len(idx) else d_buf[:0]
    for name, a in full.items():
        save_output(e, name, a.astype(np.float64))
    save_output(e, "sample_index", idx.astype(np.float64))
    save_output(e, "sample_bytes", sample.cpu().numpy().astype(np.float32))


# -------------------------------------------------------------------------------------
# the five workloads
# -------------------------------------------------------------------------------------
def run_c2(e, args, steps, warmup, full=True):
    n = args.blocks
    os.environ["ZB200_DEV_GROUP_CHUNKS"] = str(max(n, 1))   # one launch group per step: per-launch = per-step figures
    e.ctx.close()
    e.ctx = e.z.Context(e.local_rank)
    e.ctx.set_stream(e.stream.cuda_stream or e.ctx.LEGACY_DEFAULT_STREAM)   # same stream as torch's work: ordered
    d_src, T = gen_c2(e, n, e.rank * n)
    src_offs = np.arange(n + 1, dtype=np.uint64) * BLOCK
    r = measure_compress(e, d_src, src_offs, args.level, steps, warmup, e.world * n, e.rank * n, do_e2e=not args.no_e2e,
                         pageable=full and e.world == 1, parity_idx=range(64))
    out = {"metric": "compress_level%d_gzip_input_throughput" % args.level, "value": r["value"], "unit": "GiB/s",
           "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "dtype": "u8",
           "config": bench_config(n, args.level, e.world), "ratio": r["ratio"], "gpu_launches": r["gpu_launches"],
           "roofline": r["roofline"], "e2e": r.get("e2e"), "clocks": r["clocks"]}
    if "e2e_pageable" in r:
        out["e2e_pageable"] = r["e2e_pageable"]
    comp_bytes = r["comp_bytes"]
    inf_ms = r["roundtrip_inflate_ms"]
    unc = {"out_gibs": n * BLOCK / GIB / (inf_ms / 1e3), "in_gibs": comp_bytes / GIB / (inf_ms / 1e3), "ms": inf_ms,
           "note": "GPU inflate + CRC verify of this batch's own members (device-resident)"}
    if full and e.world == 1 and not args.no_e2e:
        # the reverse direction through the host-buffer call on this batch's own members
        u = measure_uncompress(e, r["_d_dst"], r["_oo"], np.full(n, BLOCK, dtype=np.uint64), max(2, steps // 4), 1,
                               do_e2e=True, h_comp=r["_h_dst"][:comp_bytes])
        ue = u["e2e"]
        unc["e2e"] = {"out_gibs": ue["out_gibs"], "in_gibs": ue["in_gibs"], "ms": ue["ms_per_step"], "h2d_bytes": comp_bytes,
                      "d2h_bytes": n * BLOCK, "h2d_ms": ue["h2d_ms"], "d2h_ms": ue["d2h_ms"], "inflate_ms": ue["inflate_ms"]}
        unc["roofline"] = u["roofline"]
    out["uncompress"] = unc
    if e.rank == 0 and not args.no_cpu:
        cores = host_threads()
        cpu, _, _ = cpu_baseline(T, n, seconds=8.0, level=args.level)
        out["cpu_baseline"] = cpu
        if full:
            b1, _, _ = cpu_baseline(T, n, seconds=2.0, threads=1, level=args.level)
            buf, bo = _c2_sample(T, 256)
            out["cpu_baselines"] = {"B1_port_1_thread": b1, "B2_port_all_threads": cpu,
                                    "B3_zlib_level1_all_threads": zlib_compress_leg(buf, bo, 1, cores),
                                    "B3_zlib_level1_1_thread": zlib_compress_leg(buf[:32 * BLOCK], bo[:33], 1, 1, 1.0),
                                    "checksums_1_thread": cpu_checksum_legs()}
            unc["cpu_baseline"] = cpu_uncompress_baseline(T)
    return out


def run_c1(e, args, reps=30, warmup=1):
    """Config 1: one file through the drop-in calls; wall-clock latency of a synchronous call."""
    import zlib
    from oracle import oracle as o
    from tests import util
    z = e.z
    raw = util.load_corpus()["alice29.txt"]
    gold_gz = util.load_golden()["alice29.txt.gz"][0]

    last = [None]   # what the last timed call returned

    def lat(f, k=reps):
        for _ in range(warmup):
            f()
        ts = []
        for _ in range(k):
            t0 = time.perf_counter()
            last[0] = f()
            ts.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(ts)), float(min(ts))

    comp = z.compress(raw, z.BestSpeed, z.dfGzip)
    assert o.uncompress(comp) == raw and zlib.decompress(comp, 31) == raw
    assert z.uncompress(comp) == raw and z.uncompress(gold_gz) == raw   # round trip bit-exact + the reference's own .gz
    c_med, c_min = lat(lambda: z.compress(raw, z.BestSpeed, z.dfGzip))
    tm_c = e.z.default_context().timing()
    if e.dump_dir:   # without the gzip header: its FNAME length is drawn at random on every call (zippy.nim:28-42)
        body = last[0][last[0].index(0, 10) + 1:]
        save_output(e, "compressed_after_header", np.frombuffer(body, dtype=np.uint8).astype(np.float32))
    u_med, u_min = lat(lambda: z.uncompress(gold_gz))
    tm_u = e.z.default_context().timing()
    if e.dump_dir:
        save_output(e, "uncompressed", np.frombuffer(last[0], dtype=np.uint8).astype(np.float32))
    oc_med, oc_min = lat(lambda: o.compress(raw, 1, o.dfGzip))
    ou_med, ou_min = lat(lambda: o.uncompress(gold_gz))
    zc_med, _ = lat(lambda: zlib.compress(raw, 1))
    zu_med, _ = lat(lambda: zlib.decompress(gold_gz, 31))
    kms = tm_u["inflate_ms"] + tm_u["verify_ms"]
    return {"workload": "C1: zippy.compress(alice29.txt, dfGzip, BestSpeed) then uncompress(alice29.txt.gz), one file per call",
            "metric": "single_file_latency", "unit": "ms", "higher_is_better": False,
            "compress_ms": c_med, "compress_min_ms": c_min, "uncompress_ms": u_med, "uncompress_min_ms": u_min,
            "value": c_med + u_med, "bytes": len(raw), "compressed_bytes": len(comp),
            "e2e": {"value": c_med + u_med, "unit": "ms", "h2d_bytes_per_step": len(raw) + len(gold_gz),
                    "d2h_bytes_per_step": len(comp) + len(raw), "note": "the drop-in calls take and return host buffers: e2e IS the value"},
            "kernel_ms": {"compress": {k: tm_c[k] for k in ("lz_ms", "huff_ms", "scan_ms", "pack_ms")},
                          "uncompress": {"inflate_ms": tm_u["inflate_ms"], "verify_ms": tm_u["verify_ms"]}},
            "roofline": roofline(e, "k_inflate", kms, len(gold_gz) + len(raw)),
            "cpu_baseline": {"value": oc_med + ou_med, "unit": "ms", "cores": 1, "kind": "port",
                             "sample": "oracle compress level 1 + uncompress of alice29, median of %d calls" % reps,
                             "compress_ms": oc_med, "uncompress_ms": ou_med, "compress_min_ms": oc_min, "uncompress_min_ms": ou_min},
            "zlib": {"compress_level1_ms": zc_med, "uncompress_ms": zu_med}, "published": PUBLISHED_C1,
            "parity": "GPU output inflated by the oracle and zlib; GPU inflate of the reference's alice29.txt.gz == original"}


def run_c3(e, args, steps, warmup):
    from tests import util
    t, z, ctx = e.torch, e.z, e.ctx
    golden = util.load_golden()
    names = sorted(nm for nm in golden if nm.endswith(".gz"))
    assert len(names) == 23
    cyc = [golden[nm][0] for nm in names]
    cyc_bytes = np.frombuffer(b"".join(cyc), dtype=np.uint8)
    n = args.members
    reps = (n + 22) // 23
    d_src = t.from_numpy(cyc_bytes.copy()).to(e.dev).repeat(reps)
    lens = np.array([len(c) for c in cyc] * reps, dtype=np.uint64)[:n]
    offs = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(lens, out=offs[1:])
    sizes, st = ctx.uncompressed_sizes_device(d_src.data_ptr(), offs, z.dfDetect)
    assert not st.any()
    r = measure_uncompress(e, d_src, offs, sizes, steps, warmup, do_e2e=not args.no_e2e)
    if e.dump_dir:
        # offsets: the output slots passed in; lengths and status: what the last timed call returned
        dump_members(e, r["_d_out"], r["_doffs"], sizes, lengths=r["_lens"], status=r["_st"])
    host = r["_d_out"][:int(r["_doffs"][23])].cpu().numpy()
    for i, nm in enumerate(names):   # byte-exact against the reference's fixtures (sha256 of the .gold / original)
        assert util.sha(host[int(r["_doffs"][i]):int(r["_doffs"][i + 1])].tobytes()) == golden[nm][1]["sha256"], nm
    # every tiling cycle equals the first (size-independent property at full size)
    cyc_out = int(r["_doffs"][23])
    full = (n // 23) * cyc_out
    v = r["_d_out"][:full].view(n // 23, cyc_out)
    assert bool((v == v[0]).all()), "tiling cycles differ"
    out = {"workload": "C3: batch uncompress of %d gzip members (the reference's 23 .gz fixtures tiled), 1 GPU" % n,
           "metric": "uncompress_gzip_input_throughput", "value": r["in_gibs"], "unit": "GiB/s", "higher_is_better": True,
           "in_gibs": r["in_gibs"], "out_gibs": r["out_gibs"], "ms_per_step": r["ms_per_step"], "in_bytes": r["in_bytes"],
           "out_bytes": r["out_bytes"], "gpu_launches": r["gpu_launches"], "roofline": r["roofline"], "e2e": r.get("e2e"),
           "clocks": r["clocks"], "parity": "first cycle sha256 == the fixtures' manifest; every cycle equal to the first; CRC + ISIZE verified on the device"}
    if not args.no_cpu:
        cores = host_threads()
        out["cpu_baseline"] = dict(cpu_uncompress_leg(cyc, int(sum(sizes[:23])), 3.0, cores), unit="GiB/s")
        out["cpu_baseline"]["value"] = out["cpu_baseline"]["in_gibs"]
        out["cpu_baselines"] = {"B1_port_1_thread": cpu_uncompress_leg(cyc, int(sum(sizes[:23])), 1.0, 1),
                                "B3_zlib_all_threads": zlib_uncompress_leg(cyc * 8, cores)}
    return out


def run_c4(e, args, steps, warmup):
    from oracle import oracle as o
    from tests import util
    t, z = e.torch, e.z
    raw = util.load_corpus()["urls.10K"]
    n = args.tiles
    d_src = t.frombuffer(bytearray(raw), dtype=t.uint8).to(e.dev).repeat(n)
    offs = np.arange(n + 1, dtype=np.uint64) * len(raw)
    r = measure_compress(e, d_src, offs, z.DefaultCompression, steps, warmup, n, 0, do_e2e=not args.no_e2e,
                         e2e_steps=max(1, steps // 2), parity_idx=range(2))
    ref = len(o.compress(raw, o.DefaultCompression, o.dfGzip))
    sz = np.diff(r["_oo"].astype(np.int64))
    assert bool((sz == sz[0]).all()), "identical tiles compressed to different sizes"
    out = {"workload": "C4: compress level=Default (dfGzip) of urls.10K x %d tiles (%.2f GiB), 1 GPU" % (n, n * len(raw) / GIB),
           "metric": "compress_default_gzip_input_throughput", "value": r["value"], "unit": "GiB/s", "higher_is_better": True,
           "ms_per_step": r["ms_per_step"], "ratio": r["ratio"], "oracle_level6_ratio": ref / float(len(raw)),
           "size_vs_reference": r["comp_bytes"] / float(ref * n), "gpu_launches": r["gpu_launches"], "roofline": r["roofline"],
           "clocks": r["clocks"], "e2e": r.get("e2e"), "parity": "round trip bit-exact on the GPU at full size; oracle + zlib inflate members; "
                                          "every tile compresses to the same bytes count"}
    if not args.no_cpu:
        cores = host_threads()
        rn = np.frombuffer(raw, dtype=np.uint8)

        def make(k):
            return np.tile(rn, k), np.arange(k + 1, dtype=np.uint64) * len(raw)

        cpu, _, _ = cpu_compress_leg(make, len(raw), o.DefaultCompression, 6.0, cores, "urls.10K tiles", max_units=4096)
        b1, _, _ = cpu_compress_leg(make, len(raw), o.DefaultCompression, 1.5, 1, "urls.10K tiles", max_units=64)
        buf, bo = make(max(cores, 2))
        out["cpu_baseline"] = cpu
        out["cpu_baselines"] = {"B1_port_1_thread": b1, "B3_zlib_level6_all_threads": zlib_compress_leg(buf, bo, 6, cores)}
    return out


def run_c5(e, args, steps, warmup):
    nb = args.c5_blocks
    first = e.rank * nb
    d_src, cls = gen_c5(e, nb, first)
    offs = np.arange(nb + 1, dtype=np.uint64) * BLOCK
    one_per_class = [int(np.nonzero(cls == k)[0][0]) for k in range(8) if (cls == k).any()]
    r = measure_compress(e, d_src, offs, 1, steps, warmup, e.world * nb, first, do_e2e=not args.no_e2e,
                         e2e_steps=max(2, steps // 2), concat=True, parity_idx=one_per_class)
    sz = np.diff(r["_oo"].astype(np.int64))
    per_class = {str(k): float(sz[cls == k].sum()) / (float((cls == k).sum()) * BLOCK) for k in range(8) if (cls == k).any()}
    inf_ms = r["roundtrip_inflate_ms"]
    out = {"workload": "C5: mixed-entropy corpus, %d x 64 KiB blocks per GPU x %d GPU(s) (8 GPUs = 64 GiB), compress level 1 "
                       "dfGzip, sizes through sharding.gather_sizes (%s), host concat at the gathered offsets in e2e"
                       % (nb, e.world, "NCCL all_gather" if e.world > 1 else "single rank"),
           "metric": "compress_level1_gzip_input_throughput", "value": r["value"], "unit": "GiB/s", "higher_is_better": True,
           "scaling": "weak", "n_gpus": e.world, "ms_per_step": r["ms_per_step"], "ratio": r["ratio"],
           "ratio_by_class": per_class, "gpu_launches": r["gpu_launches"], "roofline": r["roofline"], "e2e": r.get("e2e"),
           "clocks": r["clocks"],
           "uncompress": {"out_gibs": e.world * nb * BLOCK / GIB / (inf_ms / 1e3), "ms": inf_ms,
                          "note": "GPU inflate + verify of the shard, rank 0's time x world (device-resident)"},
           "parity": "GPU round trip bit-exact over the shard; one block per class through the oracle and zlib"}
    if e.rank == 0 and not args.no_cpu:
        from oracle import oracle as o
        cores = host_threads()
        k = 2048
        sample = d_src[:k * BLOCK].cpu().numpy()
        so = np.arange(k + 1, dtype=np.uint64) * BLOCK
        t0 = time.perf_counter()
        total, _, st = o.compress_batch(sample, so, 1, o.dfGzip, threads=cores)
        dt = time.perf_counter() - t0
        reps = int(max(1, min(16, 4.0 / max(dt, 1e-3))))
        t0 = time.perf_counter()
        for _ in range(reps):
            total, _, st = o.compress_batch(sample, so, 1, o.dfGzip, threads=cores)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": reps * k * BLOCK / GIB / dt, "unit": "GiB/s", "cores": cores, "kind": "port",
                               "sample": "first %d blocks of rank 0's shard x %d rounds, oracle level 1 gzip, %d threads, %.1f s"
                                         % (k, reps, cores, dt), "ratio": float(total) / (k * BLOCK)}
    return out


def run_large_member(e, args):
    """SURVEY 8(f-1): ONE large input.  (a) 1 GiB of text as a single gzip member of this library (64 KiB chunks
    joined by sync markers): compress and uncompress, device-resident.  (b) a FOREIGN member -- 64 MiB of text
    through system zlib level 6, no sync markers -- inflated as speculative segments, device-resident and through
    the single drop-in call; beside the oracle's single-thread inflate of the same member."""
    import zlib
    from oracle import oracle as o
    t, z, ctx = e.torch, e.z, e.ctx
    T = text_corpus()
    out = {}
    n_bytes = 1 << 30
    reps = n_bytes // len(T) + 1
    d_src = t.frombuffer(bytearray(T), dtype=t.uint8).to(e.dev).repeat(reps)[:n_bytes].contiguous()
    offs = np.array([0, n_bytes], dtype=np.uint64)
    cap = n_bytes + n_bytes // 8 + (1 << 20)
    d_dst = t.empty(cap, dtype=t.uint8, device=e.dev)
    d_back = t.empty(n_bytes, dtype=t.uint8, device=e.dev)
    oo = [None]

    def comp():
        oo[0] = ctx.compress_batch_device(d_src.data_ptr(), offs, 1, z.dfGzip, d_dst.data_ptr(), cap)

    comp()
    c_ms = timed(e, comp, 2)
    lens, st = ctx.uncompress_batch_device(d_dst.data_ptr(), oo[0], z.dfDetect, d_back.data_ptr(), offs)
    assert not st.any() and int(lens[0]) == n_bytes and t.equal(d_back, d_src)
    u_ms = timed(e, lambda: ctx.uncompress_batch_device(d_dst.data_ptr(), oo[0], z.dfDetect, d_back.data_ptr(), offs), 2)
    out["own_1GiB_member"] = {"compress_gibs": n_bytes / GIB / (c_ms / 1e3), "uncompress_out_gibs": n_bytes / GIB / (u_ms / 1e3),
                              "member_bytes": int(oo[0][1]), "kernel_launches_uncompress": int(ctx.timing()["kernel_launches"])}
    del d_src, d_dst, d_back
    raw = (T * (1 + (64 << 20) // len(T)))[:64 << 20]
    c = zlib.compressobj(6, zlib.DEFLATED, 31)
    blob = c.compress(raw) + c.flush()
    d_blob = t.frombuffer(bytearray(blob), dtype=t.uint8).to(e.dev)
    bo = np.array([0, len(blob)], dtype=np.uint64)
    do = np.array([0, len(raw)], dtype=np.uint64)
    d_out = t.empty(len(raw) + 64, dtype=t.uint8, device=e.dev)
    lens, st = ctx.uncompress_batch_device(d_blob.data_ptr(), bo, z.dfDetect, d_out.data_ptr(), do)
    assert not st.any() and int(lens[0]) == len(raw)
    assert d_out[:len(raw)].cpu().numpy().tobytes() == raw, "speculative inflate differs from the input"
    f_ms = timed(e, lambda: ctx.uncompress_batch_device(d_blob.data_ptr(), bo, z.dfDetect, d_out.data_ptr(), do), 3)
    launches = int(ctx.timing()["kernel_launches"])
    t0 = time.perf_counter()
    got = z.uncompress(blob)
    call_ms = (time.perf_counter() - t0) * 1e3
    assert got == raw
    t0 = time.perf_counter()
    o.uncompress(blob)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    out["foreign_zlib6_64MiB_member"] = {"in_bytes": len(blob), "out_bytes": len(raw), "uncompress_ms": f_ms,
                                         "uncompress_out_gibs": len(raw) / GIB / (f_ms / 1e3), "kernel_launches": launches,
                                         "single_call_ms": call_ms, "single_call_out_gibs": len(raw) / GIB / (call_ms / 1e3),
                                         "cpu_baseline": {"value": len(raw) / GIB / (cpu_ms / 1e3), "unit": "GiB/s out", "cores": 1,
                                                          "kind": "port", "sample": "oracle inflate of the same member, one call"},
                                         "parity": "byte-exact vs the input; CRC-32 + ISIZE verified on the device"}
    return out


# ======================================================================================
def run_reference(args, rank, world):
    """--impl reference: the CPU arm (oracle port on all host threads).  Rank 0 only."""
    if rank != 0:
        return
    T = text_corpus()
    cores = host_threads()
    per_step = max(6.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    if args.workload not in ("c2", "c5"):
        per_step = min(per_step, 4.0)
    times, units = [], []
    w = args.workload
    from oracle import oracle as o
    from tests import util
    extra = {}
    if w in ("c2", "c5"):
        level, unit_bytes, metric = args.level, BLOCK, "compress_level%d_gzip_input_throughput" % args.level
        cfg = bench_config(BLOCKS_PER_GPU, args.level, args.gpus)
        if w == "c5":
            cfg = {"workload": "C5 (CPU arm on text blocks of the corpus; the mixed classes need the GPU generator)"}
        for s in range(args.warmup + args.steps):
            cb, nb, dt = cpu_baseline(T, 0, seconds=per_step, threads=cores, level=level)
            if s >= args.warmup:
                times.append(dt)
                units.append(nb * unit_bytes)
        sample = "%d x 64 KiB C2 blocks per step (bounded sample of the config)" % (int(np.mean(units)) // BLOCK)
    elif w == "c4":
        raw = np.frombuffer(util.load_corpus()["urls.10K"], dtype=np.uint8)
        metric, cfg = "compress_default_gzip_input_throughput", {"workload": "C4: urls.10K tiles, level Default"}

        def make(k):
            return np.tile(raw, k), np.arange(k + 1, dtype=np.uint64) * len(raw)

        for s in range(args.warmup + args.steps):
            cb, k, dt = cpu_compress_leg(make, len(raw), o.DefaultCompression, per_step, cores, "urls.10K tiles", 4096)
            if s >= args.warmup:
                times.append(dt)
                units.append(k * len(raw))
        sample = "%d urls.10K tiles per step" % (int(np.mean(units)) // len(raw))
    elif w == "c3":
        golden = util.load_golden()
        cyc = [golden[nm][0] for nm in sorted(golden) if nm.endswith(".gz")]
        outb = sum(golden[nm][1]["len"] for nm in sorted(golden) if nm.endswith(".gz"))
        metric, cfg = "uncompress_gzip_input_throughput", {"workload": "C3: the 23 .gz fixtures tiled, batch uncompress"}
        vals = []
        for s in range(args.warmup + args.steps):
            r = cpu_uncompress_leg(cyc, outb, per_step, cores)
            if s >= args.warmup:
                vals.append(r)
        val = float(np.mean([v["in_gibs"] for v in vals]))
        extra = {"out_gibs": float(np.mean([v["out_gibs"] for v in vals]))}
        times, units, sample = [1.0], [val * GIB], vals[-1]["sample"]
    else:  # c1
        raw = util.load_corpus()["alice29.txt"]
        gz = util.load_golden()["alice29.txt.gz"][0]
        ts = []
        for s in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            c = o.compress(raw, 1, o.dfGzip)
            o.uncompress(gz)
            if s >= args.warmup:
                ts.append((time.perf_counter() - t0) * 1e3)
        val = float(np.median(ts))
        out = {"impl": "reference", "metric": "single_file_latency", "value": val, "unit": "ms", "n_gpus": args.gpus,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": val, "higher_is_better": False, "scaling": "weak",
               "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": {"workload": "C1: alice29.txt compress + uncompress"},
               "cpu_baseline": {"value": val, "unit": "ms", "cores": 1, "kind": "port", "sample": "median of %d calls" % args.steps},
               "e2e": {"value": val, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(out))
        return
    val = sum(units) / GIB / sum(times)
    out = {"impl": "reference", "metric": metric, "value": val, "unit": "GiB/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
           "cpu_baseline": {"value": val, "unit": "GiB/s", "cores": cores, "kind": "port",
                            "sample": sample + ", oracle port of zippy (Nim unavailable: the reference cannot be compiled "
                                      "here; built -O3 -march=x86-64-v3 with the PCLMUL CRC-32 / SSSE3 Adler-32 paths), "
                                      "all %d host threads" % cores},
           "e2e": {"value": val, "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    out.update(extra)
    if w == "c2":
        out["uncompress"] = {"cpu_baseline": cpu_uncompress_baseline(T, seconds=3.0, threads=cores)}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--blocks", type=int, default=BLOCKS_PER_GPU, help="c2: 64 KiB blocks per GPU (default = config)")
    ap.add_argument("--members", type=int, default=C3_MEMBERS, help="c3: gzip members")
    ap.add_argument("--tiles", type=int, default=C4_TILES, help="c4: urls.10K tiles")
    ap.add_argument("--c5-blocks", type=int, default=C5_BLOCKS_PER_GPU, help="c5: 64 KiB blocks per GPU")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="c2 only: skip the c1/c3/c4/c5 summaries")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--level", type=int, default=1)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed path's outputs of its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the GPU path's outputs (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    e = make_env(args)
    clocks = ClockSampler(e.local_rank)
    clocks.start()
    clocks.mark()
    e.clocks = clocks
    e.last_clocks = None
    e.dump_dir = args.dump_outputs   # the selected workload's outputs only, not the extras'
    w = args.workload
    extras = {}
    if w == "c2":
        out = run_c2(e, args, args.steps, args.warmup)
        e.dump_dir = None
        main_clk = out.pop("clocks")
        if not args.no_extras:
            xs = max(2, min(args.steps, 3))
            if e.world == 1:
                if not args.no_e2e:
                    extras["pcie"] = pcie_peaks(e)
                for name, fn in (("c1", lambda: run_c1(e, args)), ("c3", lambda: run_c3(e, args, xs, 3)),
                                 ("c4", lambda: run_c4(e, args, xs, 3)), ("c5", lambda: run_c5(e, args, xs, 3)),
                                 ("large_member", lambda: run_large_member(e, args)),
                                 ("checksums", lambda: run_checksums(e, args))):
                    e.torch.cuda.empty_cache()
                    try:
                        extras[name] = strip(fn())
                    except Exception as ex:   # an extra must not take the headline line down with it
                        extras[name] = {"error": repr(ex)}
            else:
                e.torch.cuda.empty_cache()
                extras["c5"] = strip(run_c5(e, args, xs, 3))
    else:
        fn = {"c1": lambda: run_c1(e, args, args.steps, args.warmup), "c3": lambda: run_c3(e, args, args.steps, args.warmup),
              "c4": lambda: run_c4(e, args, args.steps, args.warmup), "c5": lambda: run_c5(e, args, args.steps, args.warmup)}[w]
        out = fn()
        out.setdefault("scaling", "weak")
        out["dtype"] = "u8"
        out["config"] = {"workload": out.pop("workload")}
        if "ms_per_step" not in out:
            out["ms_per_step"] = out["value"]
        if w != "c5" and not args.no_e2e:
            extras["pcie"] = pcie_peaks(e)
        main_clk = out.pop("clocks", None) or clocks.snapshot()
    clocks.finish()
    if e.rank == 0:
        line = {"metric": out.pop("metric"), "value": out.pop("value"), "unit": out.pop("unit"), "n_gpus": e.world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": out.pop("ms_per_step"),
                "higher_is_better": out.pop("higher_is_better"), "scaling": out.pop("scaling"), "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": out.pop("config"), "clocks": main_clk, "numa": e.numa}
        line.update(strip(out))
        line.setdefault("cpu_baseline", None)
        if extras:
            line["extras"] = extras
        print(json.dumps(line))
    if e.world > 1:
        e.dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- the hot path of rorosen/zeekstd (per-frame compress + decompress of a seekable archive) on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

One STEP = compress a buffer into a seekable archive AND decompress that archive again (one pass of the hot path in both
directions); `value` = uncompressed GiB moved per second over the step (2 x buffer / step time).

N = 1 (BASELINE.json configs[1]): a 1 GiB Silesia-like mix (text = dickens.txt slices), 2 MiB frames, level 1, inputs
resident in HBM (CUDA events around every kernel of both calls).  `e2e` is the same step through the host-pointer C ABI
(zk_compress_frames / zk_decompress_frames: pinned host buffers, H2D + D2H inside the timed region).  `config4_one_gpu`
adds the level-3 + checksum figure of configs[3] on one GPU (what the multi-GPU line below divides).

N > 1 (BASELINE.json configs[3], SURVEY.md 8e): STRONG scaling of ONE root-held buffer (16 GiB mixed-entropy, 2 MiB
frames, level 3, checksum on).  Inside the timed region: the root scatters frame ranges over NCCL, every rank
compresses its frames, all-gather of the frame sizes, variable gather of the archive to the root; then the archive is
scattered by seek-table offsets, decoded, and the output gathered to the root (zeekstd_b200/parallel.py: chunked and
pipelined, two communicators).  `per_rank` breaks the step down (codec vs exchange), `limiting` names the slower piece.
`weak` keeps the exchange-free figure (every rank its own 1 GiB of configs[1]); `e2e` is the host-buffer step of
configs[1] per rank (data that originates on the host goes H2D per GPU, no NCCL -- SURVEY.md 8e).

--impl reference times the reference's own CPU path: libzstd driven through zeekstd's call sequence
(oracle/libzstd_driver.c; the Rust crate itself cannot be built in this image -- no cargo, no network) on the SAME
bytes (the generator is counter-based: identical on CPU and GPU), frames spread over every host thread; what one thread
reaches (zeekstd itself is single-threaded) is reported beside it.  Both arms report the MEAN over the timed steps.
`roofline.traffic` comes from the committed ncu capture named in `traffic_source`: a bench value is never taken under a
profiler.

--dump-outputs DIR writes, after the timed steps, what the last timed step handed its caller (rank 0's, at N > 1): archive.npy and
output.npy (the compressed archive and the restored bytes, as float32, at fixed seeded positions when longer than 4 Mi bytes) and
c_sizes.npy / d_sizes.npy (the seek table, float64).  The inputs depend only on the arguments, so two builds of the project can be
compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAME = 2 << 20
LEVEL = 1
WORKLOAD_BYTES = int(os.environ.get("ZK_BENCH_BYTES", str(1 << 30)))
C4_BYTES = int(os.environ.get("ZK_BENCH_C4_BYTES", str(16 << 30)))         # configs[3]: 16 GiB on the root
C4_ONE_GPU_BYTES = int(os.environ.get("ZK_BENCH_C4_ONE_BYTES", str(4 << 30)))
C4_REF_BYTES = int(os.environ.get("ZK_BENCH_C4_REF_BYTES", str(4 << 30)))   # bounded sample for the CPU arm at N > 1
C4_LEVEL, C4_SEED = 3, 20260925
SEED = 20260924
METRIC = "GiB/s compress + decompress (2 MiB frames)"
DUMP_SEED = 20261017
DUMP_SAMPLE = 1 << 22                      # bytes kept of each byte stream: 2 x 16 MiB of float32 in all
KERNEL_NAMES = ["zk_scan_kernel", "zk_seq_kernel", "zk_huf_kernel", "zk_exec_kernel", "zk_xxh64_kernel", "zk_match_kernel",
                "zk_entropy_enc_kernel", "zk_frame_*_kernels"]
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "traffic_r2.json")


def workload_c1():
    from zeekstd_b200 import corpus
    return f"silesia-mix {WORKLOAD_BYTES >> 20} MiB (configs[1]); text = {corpus.text_source()}"


def workload_c4(nbytes):
    from zeekstd_b200 import corpus
    return f"mixed-entropy {nbytes >> 20} MiB (configs[3]); text = {corpus.text_source()}"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def whole_direction(n_plain, n_comp, c_ms, d_ms, n_gpus):
    """HBM roofline of each whole direction (not only the dominant kernel): algorithmic bytes = plain + compressed bytes of the job, over the
    direction's device time, against n_gpus x the measured peak.  Pure arithmetic on numbers the line already carries."""
    try:
        peak, _ = peaks()
        alg = float(n_plain + n_comp)
        c, d = alg / (c_ms / 1e3) / 1e9, alg / (d_ms / 1e3) / 1e9
        return {"algorithmic_bytes": int(alg), "compress_GBps": round(c, 1), "decompress_GBps": round(d, 1),
                "compress_frac": round(c / (peak * n_gpus), 5), "decompress_frac": round(d / (peak * n_gpus), 5), "peak_GBps": peak * n_gpus}
    except Exception:                                               # never worth losing the line for
        return None


class ClockSampler(threading.Thread):
    """samples SM clock / throttle reasons of one GPU during the timed region (NVML; nvidia-smi semantics)"""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        self.stop_flag = True
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def gen_mix(nbytes: int, seed: int, mix=None, device="cpu"):
    """the workload generator, in 1 GiB slabs (bounds the generator's scratch); identical bytes on every device"""
    import torch
    from zeekstd_b200 import corpus
    slab = 1 << 30
    parts = [corpus.make_mix(min(slab, nbytes - o), seed=seed + (o >> 30), mix=mix, device=device) for o in range(0, nbytes, slab)]
    return parts[0] if len(parts) == 1 else torch.cat(parts)


def byte_sample(buf, n: int) -> np.ndarray:
    """buf[:n] (a uint8 tensor) as float32: every byte, or DUMP_SAMPLE bytes at seeded positions that depend only on n"""
    import torch
    idx = np.arange(n) if n <= DUMP_SAMPLE else np.sort(np.random.default_rng(DUMP_SEED).integers(0, n, DUMP_SAMPLE))
    return buf[torch.from_numpy(idx).to(buf.device)].cpu().numpy().astype(np.float32)


def dump_outputs(out_dir: str, archive, archive_len: int, c_sizes, d_sizes, output, output_len: int) -> None:
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"archive": byte_sample(archive, archive_len), "output": byte_sample(output, output_len),
              "c_sizes": np.asarray(c_sizes, dtype=np.float64), "d_sizes": np.asarray(d_sizes, dtype=np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_reference(data: np.ndarray, threads: int, level: int = LEVEL, checksum: bool = False):
    """the reference path on the host cores: libzstd through zeekstd's call sequence -> (seconds compress, seconds decompress, ratio)"""
    from oracle import oracle as O
    t0 = time.perf_counter()
    frames, cs, ds = O.ref_compress_frames(data, FRAME, level, checksum, threads=threads)
    t1 = time.perf_counter()
    comp = np.frombuffer(b"".join(frames), dtype=np.uint8)
    co = np.zeros(len(cs) + 1, dtype=np.uint64); co[1:] = np.cumsum(cs)
    do = np.zeros(len(ds) + 1, dtype=np.uint64); do[1:] = np.cumsum(ds)
    t2 = time.perf_counter()
    out, sizes = O.ref_decompress_frames(comp, co, do, threads=threads)
    t3 = time.perf_counter()
    assert all(s == d for s, d in zip(sizes, ds))
    return t1 - t0, t3 - t2, data.size / sum(cs)


def cpu_rates(data: np.ndarray, threads: int, reps: int, level: int = LEVEL, checksum: bool = False):
    """mean over `reps` passes -> (GiB/s step, compress, decompress, ratio)"""
    tc = td = 0.0
    for _ in range(reps):
        a, b, ratio = cpu_reference(data, threads, level, checksum)
        tc += a; td += b
    gib = data.size / 2**30 * reps
    return 2 * gib / (tc + td), gib / tc, gib / td, ratio


def single_thread_note(data: np.ndarray, level: int, checksum: bool):
    v = cpu_rates(data, 1, 1, level, checksum)
    return {"cores": 1, "value": round(v[0], 4), "compress_GiBps": round(v[1], 4), "decompress_GiBps": round(v[2], 4),
            "sample": f"{data.size >> 20} MiB", "note": "what zeekstd's own single-threaded Encoder/Decoder reaches"}


L2_NOTE = "GPU arm: a 256 MiB buffer is written between timed iterations and the inputs exceed the 126 MB L2"
EXCHANGE_C4 = ("GPU arm: NCCL inside the timed region -- scatter input -> compress -> all_gather(frame sizes) -> gather archive to root; "
               "scatter archive -> decompress -> gather output to root (chunked, pipelined, two communicators)")


def config_c1(n):
    """the SAME dict in both arms (the driver compares them)"""
    return {"workload": workload_c1(), "frame_size": FRAME, "level": LEVEL, "checksum": False, "bytes_per_gpu": n, "step": "compress+decompress",
            "l2": L2_NOTE, "exchange": "none"}


def config_c4(nbytes, world):
    return {"workload": workload_c4(nbytes), "frame_size": FRAME, "level": C4_LEVEL, "checksum": True, "bytes_total": nbytes, "step": "compress+decompress",
            "parallelism": f"frames sharded over {world} GPUs, root-held buffer", "l2": L2_NOTE, "exchange": EXCHANGE_C4}


# ================================================================================================ reference arm
def main_reference(args, rank, world, ncores):
    if rank != 0:
        return 0
    import torch
    from oracle import oracle as O
    W = max(args.warmup, 0); K = args.steps
    dev = "cuda" if torch.cuda.is_available() else "cpu"        # generation only (same bytes either way); nothing of ours runs here
    if args.gpus <= 1:
        data = gen_mix(WORKLOAD_BYTES, SEED, device=dev).cpu().numpy()
        level, ck, cfg = LEVEL, False, config_c1(WORKLOAD_BYTES)
        sample = f"the whole {WORKLOAD_BYTES >> 20} MiB workload per step"
        scaling = "weak"
    else:
        from zeekstd_b200 import corpus
        nb = min(C4_BYTES, C4_REF_BYTES)
        data = gen_mix(nb, C4_SEED, corpus.CLASS_MIX_MIXED, device=dev).cpu().numpy()
        level, ck, cfg = C4_LEVEL, True, config_c4(C4_BYTES, args.gpus)
        sample = f"the first {nb >> 30} GiB of the {C4_BYTES >> 30} GiB workload per step (bounded so the run ends within minutes)"
        scaling = "strong"
    for _ in range(min(W, 2)):
        cpu_reference(data[: 256 << 20], ncores, level, ck)
    t0 = time.perf_counter()
    v = cpu_rates(data, ncores, K, level, ck)
    dt = (time.perf_counter() - t0) / K
    one = single_thread_note(data[: min(data.size, 128 << 20)], level, ck)
    line = {"metric": METRIC, "value": round(v[0], 4), "unit": "GiB/s", "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": round(dt * 1e3, 2),
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic", "impl": "reference",
            "config": cfg, "statistic": "mean over the timed steps",
            "compress_GiBps": round(v[1], 4), "decompress_GiBps": round(v[2], 4), "ratio": round(v[3], 4),
            "cpu_baseline": {"value": round(v[0], 4), "unit": "GiB/s", "cores": ncores, "kind": "reference",
                             "sample": f"{sample}; libzstd {O.libzstd_version()} through the reference's call sequence (oracle/libzstd_driver.c), "
                                       f"frames spread over {ncores} host threads",
                             "single_thread": one},
            "e2e": {"value": round(v[0], 4), "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)
    return 0


# ================================================================================================ our arm, shared pieces
class Rig:
    """one rank's GPU context + the two measurements every N shares (device-resident step, host-pointer step)"""

    def __init__(self, local):
        import torch
        import zeekstd_b200 as zk
        from zeekstd_b200 import _native as N
        self.torch, self.N = torch, N
        self.lib = N.load()
        self.ctx = zk.Context(local, self.lib)
        self.dev = torch.device("cuda", local)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)          # > 126 MB L2: written between steps

    def device_step_fn(self, x, level, checksum):
        torch, N, lib, ctx = self.torch, self.N, self.lib, self.ctx
        n = x.numel()
        src = torch.cat([x, torch.zeros(64, dtype=torch.uint8, device=self.dev)])
        cap = lib.zk_compress_bound(n, FRAME)
        comp = torch.zeros(cap + 64, dtype=torch.uint8, device=self.dev)
        back = torch.zeros(n + 64, dtype=torch.uint8, device=self.dev)
        nfmax = n // FRAME + 2
        cs = np.zeros(nfmax, dtype=np.uint32); ds = np.zeros(nfmax, dtype=np.uint32)
        nf = ctypes.c_uint32(); dl = ctypes.c_size_t()
        torch.cuda.synchronize()          # the codec runs on its own (non-blocking) stream: the buffers above must be complete before it reads them

        def step():
            rc = lib.zk_compress_frames_dev(ctx._h, src.data_ptr(), n, FRAME, level, int(checksum), comp.data_ptr(), cap, cs.ctypes.data_as(N.u32p),
                                            ds.ctypes.data_as(N.u32p), nfmax, ctypes.byref(nf), ctypes.byref(dl), None)
            assert rc == 0, rc
            t_c = ctx.last_device_ms
            k = nf.value
            co = np.zeros(k + 1, dtype=np.uint64); co[1:] = np.cumsum(cs[:k]); do = np.zeros(k + 1, dtype=np.uint64); do[1:] = np.cumsum(ds[:k])
            rc = lib.zk_decompress_frames_dev(ctx._h, comp.data_ptr(), co.ctypes.data_as(N.u64p), do.ctypes.data_as(N.u64p), k, back.data_ptr(), int(checksum), None, None)
            assert rc == 0, rc
            return t_c, ctx.last_device_ms, int(co[-1])
        step.comp, step.back, step.cs, step.ds, step.nf = comp, back, cs, ds, nf
        return step

    def timed_device(self, x, level, checksum, warmup, steps, dist=None):
        """-> (compress ms/step, decompress ms/step, compressed bytes), device time, L2 flushed between steps"""
        torch = self.torch
        step = self.device_step_fn(x, level, checksum)
        for _ in range(max(warmup, 3)):
            self.flush.fill_(1)
            step()
        assert torch.equal(step.back[: x.numel()], x), "round trip mismatch"
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        tc = td = 0.0; clen = 0
        for _ in range(steps):
            self.flush.fill_(1); torch.cuda.synchronize()
            a, b, clen = step()
            tc += a; td += b
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        self.last_step = step
        return tc / steps, td / steps, clen

    def timed_host(self, x, level, checksum, steps, dist=None):
        """the same step through the host-pointer C ABI with pinned buffers -> (s compress, s decompress, compressed bytes)"""
        torch, N, lib, ctx = self.torch, self.N, self.lib, self.ctx
        n = x.numel()
        cap = lib.zk_compress_bound(n, FRAME)
        h_src = torch.empty(n, dtype=torch.uint8).pin_memory(); h_src.copy_(x.cpu())
        h_comp = torch.empty(cap + 64, dtype=torch.uint8).pin_memory()
        h_back = torch.empty(n + 64, dtype=torch.uint8).pin_memory()
        nfmax = n // FRAME + 2
        cs = np.zeros(nfmax, dtype=np.uint32); ds = np.zeros(nfmax, dtype=np.uint32)
        nf = ctypes.c_uint32(); dl = ctypes.c_size_t()

        def step():
            t0 = time.perf_counter()
            rc = lib.zk_compress_frames(ctx._h, h_src.data_ptr(), n, FRAME, level, int(checksum), h_comp.data_ptr(), cap, cs.ctypes.data_as(N.u32p),
                                        ds.ctypes.data_as(N.u32p), nfmax, ctypes.byref(nf), ctypes.byref(dl))
            assert rc == 0, rc
            t1 = time.perf_counter()
            k = nf.value
            co = np.zeros(k + 1, dtype=np.uint64); co[1:] = np.cumsum(cs[:k]); do = np.zeros(k + 1, dtype=np.uint64); do[1:] = np.cumsum(ds[:k])
            t2 = time.perf_counter()
            rc = lib.zk_decompress_frames(ctx._h, h_comp.data_ptr(), co.ctypes.data_as(N.u64p), do.ctypes.data_as(N.u64p), k, h_back.data_ptr(), int(checksum), None)
            assert rc == 0, rc
            return t1 - t0, time.perf_counter() - t2, int(co[-1])

        for _ in range(2):
            step()
        if dist:
            dist.barrier()
        ec = ed = 0.0; clen = 0
        for _ in range(steps):
            a, b, clen = step()
            ec += a; ed += b
        assert torch.equal(h_back[:n], h_src), "host round trip mismatch"
        return ec / steps, ed / steps, clen


def c4_host_leg(parallel, codec, xr, nb, frame, level, dev, rank, steps, sync, pin):
    """e2e of the configs[3] workload at N > 1: the root's input, archive and output live in (pinned) HOST memory; every step copies the input
    up, runs the sharded passes, and copies the archive / the output down (copies not overlapped with the exchange: the root's PCIe link carries
    every byte).  All ranks first agree that the root got its host buffers, so that nobody waits in a collective the root never enters.
    -> the e2e dict on the root, None elsewhere or when the leg could not run.  (Runs on CPU tensors over gloo too: tests/test_parallel_gloo.py.)"""
    import torch
    import torch.distributed as dist
    gib = 2.0**30
    ok = torch.ones(1, dtype=torch.int32, device=dev)
    h_x = h_arc = h_out = None
    if rank == 0:
        try:
            h_x = torch.empty(nb, dtype=torch.uint8, pin_memory=pin); h_x.copy_(xr[:nb])
            h_arc = torch.empty(nb, dtype=torch.uint8, pin_memory=pin)       # (torch's pinned allocator rounds up to a power of two: not the bound)
            h_out = torch.empty(nb, dtype=torch.uint8, pin_memory=pin)
        except (RuntimeError, MemoryError) as e:
            sys.stderr.write(f"bench: no host buffers for the configs[3] e2e leg ({e}); keeping the per-rank figure\n")
            ok.zero_()
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if int(ok.item()) != 1:
        return None
    tc_w = td_w = 0.0
    clen_e = 0
    for it in range(steps + 1):                                          # first pass untimed
        sync(); dist.barrier()
        t0 = time.perf_counter()
        if rank == 0:
            xr[:nb].copy_(h_x, non_blocking=True)
        frames, cs, ds = parallel.sharded_compress(codec, xr, nb, frame, level, True, device=dev)
        clen_e = int(np.sum(cs))
        if clen_e > nb:                                                  # every rank holds the same sizes: a common decision
            return None
        if rank == 0:
            h_arc[:clen_e].copy_(frames[:clen_e], non_blocking=True)
        sync(); dist.barrier()
        t1 = time.perf_counter()
        if rank == 0:
            frames[:clen_e].copy_(h_arc[:clen_e], non_blocking=True)
        back = parallel.sharded_decompress(codec, frames, cs, ds, True, device=dev, frame_size=frame)
        if rank == 0:
            h_out.copy_(back[:nb], non_blocking=True)
        sync(); dist.barrier()
        t2 = time.perf_counter()
        if it:
            tc_w += t1 - t0; td_w += t2 - t1
        del frames, back
    tw = torch.tensor([tc_w / steps, td_w / steps], dtype=torch.float64, device=dev)
    dist.all_reduce(tw, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    if not torch.equal(h_out, h_x):
        sys.stderr.write("bench: configs[3] host round trip MISMATCH; the e2e leg is dropped\n")
        return None
    ec4, ed4 = float(tw[0]), float(tw[1])
    return {"value": round(2 * (nb / gib) / (ec4 + ed4), 3), "unit": "GiB/s", "h2d_bytes_per_step": int(nb + clen_e), "d2h_bytes_per_step": int(clen_e + nb),
            "compress_GiBps": round(nb / gib / ec4, 3), "decompress_GiBps": round(nb / gib / ed4, 3), "steps": steps,
            "api": "pinned host buffers on the root <-> root GPU <-> parallel.sharded_compress / sharded_decompress (NCCL); wall clock, copies not overlapped "
                   "with the exchange -- the root's PCIe link carries every byte, so this figure does not grow with N"}


def roofline_block(rig, alg_bytes, n):
    lib, ctx = rig.lib, rig.ctx
    kms = (ctypes.c_float * 8)(); kcnt = (ctypes.c_uint32 * 8)()
    lib.zk_ctx_profile_read(ctx._h, kms, kcnt)
    peak, peak_src = peaks()
    per = [float(kms[i]) / max(1, int(kcnt[i])) for i in range(8)]
    dom = int(np.argmax(per))
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(TRAFFIC_FILE))
        if n == (1 << 30) and KERNEL_NAMES[dom] in tj["bytes_per_launch"]:
            traffic, traffic_src = tj["bytes_per_launch"][KERNEL_NAMES[dom]], tj["source"]
    except (OSError, ValueError, KeyError):
        pass
    achieved = alg_bytes / (per[dom] / 1e3) / 1e9 if per[dom] > 0 else 0.0
    return {"bound": "hbm", "kernel": KERNEL_NAMES[dom], "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 5),
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": int(alg_bytes),
            "kernel_ms": {KERNEL_NAMES[i]: round(per[i], 3) for i in range(8) if kcnt[i]},
            "note": "the path is bound by serial entropy / match dependencies, not by HBM (SURVEY.md 8d)"}


def cpu_baseline_block(x_cpu: np.ndarray, ncores, level, checksum, what):
    from oracle import oracle as O
    allc = cpu_rates(x_cpu, ncores, 1, level, checksum)
    return {"value": round(allc[0], 4), "unit": "GiB/s", "cores": ncores, "kind": "reference", "compress_GiBps": round(allc[1], 4),
            "decompress_GiBps": round(allc[2], 4), "ratio": round(allc[3], 4),
            "sample": f"{what}, one pass; libzstd {O.libzstd_version()} through the reference's call sequence (oracle/libzstd_driver.c), frames spread over {ncores} host threads",
            "single_thread": single_thread_note(x_cpu[: min(x_cpu.size, 128 << 20)], level, checksum)}


# ================================================================================================ our arm
def main_ours(args, rank, world, local, ncores):
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: zeekstd_b200 has no CPU fallback"}), flush=True)
        return 2
    from zeekstd_b200 import corpus
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))   # a hang must fail fast
    rig = Rig(local)
    lib, ctx, dev = rig.lib, rig.ctx, rig.dev
    W, K = max(args.warmup, 3), args.steps
    gib = 2.0**30

    # ---------------------------------------------------------------- configs[1] on this rank's GPU (headline at N = 1, `weak` at N > 1)
    n = WORKLOAD_BYTES
    x = gen_mix(n, SEED + rank, device=dev)                                     # unique per rank
    launches0 = ctx.kernel_launches
    lib.zk_ctx_profile(ctx._h, 1)
    sampler = ClockSampler(local); sampler.start()
    tc_ms, td_ms, clen = rig.timed_device(x, LEVEL, False, W, K, dist)
    clocks = sampler.result()
    launches = ctx.kernel_launches - launches0
    roof = roofline_block(rig, n + clen, n) if rank == 0 else None
    lib.zk_ctx_profile(ctx._h, 0)
    if args.dump_outputs and world == 1:
        s = rig.last_step
        dump_outputs(args.dump_outputs, s.comp, clen, s.cs[: s.nf.value], s.ds[: s.nf.value], s.back, n)
    t = torch.tensor([tc_ms, td_ms], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                                # device time, max over ranks
    tc_ms, td_ms = float(t[0]), float(t[1])
    weak_value = world * 2 * (n / gib) / ((tc_ms + td_ms) / 1e3)
    # ---- e2e through the host-pointer C ABI (H2D + D2H inside the timed region)
    ec_s, ed_s, clen_h = rig.timed_host(x, LEVEL, False, K, dist)
    te = torch.tensor([ec_s, ed_s], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    ec_s, ed_s = float(te[0]), float(te[1])
    e2e = {"value": round(world * 2 * (n / gib) / (ec_s + ed_s), 3), "unit": "GiB/s", "h2d_bytes_per_step": int(n + clen_h), "d2h_bytes_per_step": int(clen_h + n),
           "compress_GiBps": round(world * (n / gib) / ec_s, 3), "decompress_GiBps": round(world * (n / gib) / ed_s, 3),
           "api": "zk_compress_frames + zk_decompress_frames (pinned host buffers)" + ("; every rank its own 1 GiB of configs[1]" if world > 1 else "")}

    if world == 1:
        # ---- configs[3] shape on one GPU: level 3 + checksum (fused into the codec kernels), device-resident
        nb = min(C4_BYTES, C4_ONE_GPU_BYTES)
        x4 = gen_mix(nb, C4_SEED, corpus.CLASS_MIX_MIXED, device=dev)
        c4c, c4d, c4len = rig.timed_device(x4, C4_LEVEL, True, 3, max(2, K // 2))
        c4 = {"config": config_c4(nb, 1), "value": round(2 * (nb / gib) / ((c4c + c4d) / 1e3), 3), "compress_GiBps": round(nb / gib / (c4c / 1e3), 3),
              "decompress_GiBps": round(nb / gib / (c4d / 1e3), 3), "ratio": round(nb / c4len, 4)}
        del x4, rig.last_step
        torch.cuda.empty_cache()
        line = {"metric": METRIC, "value": round(weak_value, 3), "unit": "GiB/s", "n_gpus": 1, "steps": K, "warmup": W,
                "ms_per_step": round(tc_ms + td_ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config_c1(n),
                "statistic": "mean over the timed steps",
                "compress_GiBps": round(n / gib / (tc_ms / 1e3), 3), "decompress_GiBps": round(n / gib / (td_ms / 1e3), 3),
                "ratio": round(n / clen, 4), "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e, "roofline": roof,
                "roofline_whole_direction": whole_direction(n, clen, tc_ms, td_ms, 1), "config4_one_gpu": c4,
                "cpu_baseline": cpu_baseline_block(x.cpu().numpy(), ncores, LEVEL, False, f"the {n >> 20} MiB workload")}
        print(json.dumps(line), flush=True)
        return 0

    # ---------------------------------------------------------------- N > 1: configs[3], strong scaling, exchange inside the timed region
    from zeekstd_b200 import parallel
    parallel.groups(dev)                       # creates AND exercises the communicators before anything is in flight
    weak = {"value": round(weak_value, 3), "unit": "GiB/s", "scaling": "weak", "compress_GiBps": round(world * n / gib / (tc_ms / 1e3), 3),
            "decompress_GiBps": round(world * n / gib / (td_ms / 1e3), 3), "config": config_c1(n)}
    del x
    torch.cuda.empty_cache()
    nb = C4_BYTES
    codec = parallel.DeviceCodec(ctx)
    xr = None
    if rank == 0:
        xr = codec.empty(nb, dev)
        for o in range(0, nb, 1 << 30):
            xr[o: o + min(1 << 30, nb - o)] = corpus.make_mix(min(1 << 30, nb - o), seed=C4_SEED + (o >> 30), mix=corpus.CLASS_MIX_MIXED, device=dev)
        xr[nb:] = 0
        torch.cuda.empty_cache()
    stats = {}

    def step(collect=None):
        frames, cs, ds = parallel.sharded_compress(codec, xr, nb, FRAME, C4_LEVEL, True, device=dev, stats=collect)
        back = parallel.sharded_decompress(codec, frames, cs, ds, True, device=dev, stats=collect, frame_size=FRAME)
        return frames, cs, back

    for _ in range(W):
        rig.flush.fill_(1)
        frames, cs, back = step()
    if rank == 0:
        assert torch.equal(back[:nb], xr[:nb]), "sharded round trip mismatch"
    del frames, back
    launches0 = ctx.kernel_launches
    sampler = ClockSampler(local); sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    dist.barrier(); torch.cuda.synchronize()
    tcs = tds = 0.0
    acc = {}
    for it in range(K):
        rig.flush.fill_(1); torch.cuda.synchronize(); dist.barrier()
        st = {}
        ev[0].record()
        frames, cs, ds = parallel.sharded_compress(codec, xr, nb, FRAME, C4_LEVEL, True, device=dev, stats=st)
        ev[1].record()
        back = parallel.sharded_decompress(codec, frames, cs, ds, True, device=dev, stats=st, frame_size=FRAME)
        ev[2].record(); torch.cuda.synchronize()
        tcs += ev[0].elapsed_time(ev[1]); tds += ev[1].elapsed_time(ev[2])
        for k_, v_ in st.items():
            acc[k_] = acc.get(k_, 0.0) + float(v_)
        clen4 = int(np.sum(cs))
        if args.dump_outputs and rank == 0 and it == K - 1:
            dump_outputs(args.dump_outputs, frames, clen4, cs, ds, back, nb)
        del frames, back
    torch.cuda.synchronize(); dist.barrier()
    clocks4 = sampler.result()
    e2e4 = c4_host_leg(parallel, codec, xr, nb, FRAME, C4_LEVEL, dev, rank, max(1, min(2, K)), torch.cuda.synchronize, True)
    if e2e4 is not None:
        e2e4["per_rank_configs1"] = e2e
    launches4 = ctx.kernel_launches - launches0
    t4 = torch.tensor([tcs / K, tds / K], dtype=torch.float64, device=dev)
    dist.all_reduce(t4, op=dist.ReduceOp.MAX)
    c_ms, d_ms = float(t4[0]), float(t4[1])
    keys = ["compress_total_ms", "compress_until_codec_done_ms", "compress_codec_ms", "compress_gather_ms", "decompress_total_ms", "decompress_codec_ms",
            "decompress_wait_ms", "compress_chunks", "chunk_frames"]
    mine = torch.tensor([acc.get(k_, 0.0) / K for k_ in keys] + [float(launches4)], dtype=torch.float64, device=dev)
    allr = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(allr, mine)
    if rank != 0:
        dist.destroy_process_group()
        return 0
    per_rank = [dict({"rank": r}, **{k_: round(float(allr[r][i]), 3) for i, k_ in enumerate(keys)}) for r in range(world)]
    value = 2 * (nb / gib) / ((c_ms + d_ms) / 1e3)
    codec_c = max(p["compress_codec_ms"] for p in per_rank); codec_d = max(p["decompress_codec_ms"] for p in per_rank)
    exch_c, exch_d = c_ms - codec_c, d_ms - codec_d
    limiting = (f"compress: slowest rank's codec {codec_c:.1f} ms of {c_ms:.1f} ms (scatter wait + size all-gather + archive gather {exch_c:.1f} ms); "
                f"decompress: slowest rank's codec {codec_d:.1f} ms of {d_ms:.1f} ms (exchange not hidden {exch_d:.1f} ms) -> "
                + ("the exchange through the root's NVLink (scatter of the input / gather of the output)" if exch_c + exch_d > 0.5 * (codec_c + codec_d)
                   else "the codec on the slowest rank"))
    # one GPU, same workload shape, no exchange (bounded sample) -- what the strong-scaling figure divides
    nb1 = min(nb, C4_ONE_GPU_BYTES)
    one_c, one_d, _ = rig.timed_device(xr[:nb1].clone(), C4_LEVEL, True, 2, 2)
    one_gpu = {"value": round(2 * (nb1 / gib) / ((one_c + one_d) / 1e3), 3), "compress_GiBps": round(nb1 / gib / (one_c / 1e3), 3),
               "decompress_GiBps": round(nb1 / gib / (one_d / 1e3), 3), "sample": f"first {nb1 >> 30} GiB of the same buffer on rank 0, device-resident, no exchange"}
    sample = xr[: min(nb, C4_REF_BYTES // 2)].cpu().numpy()
    line = {"metric": METRIC, "value": round(value, 3), "unit": "GiB/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": round(c_ms + d_ms, 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config_c4(nb, world),
            "statistic": "mean over the timed steps; device time (CUDA events), max over ranks",
            "compress_GiBps": round(nb / gib / (c_ms / 1e3), 3), "decompress_GiBps": round(nb / gib / (d_ms / 1e3), 3), "ratio": round(nb / clen4, 4),
            "per_rank": per_rank, "limiting": limiting, "one_gpu_same_workload": one_gpu, "weak": weak,
            "gpu_launches": int(sum(float(a[-1]) for a in allr)), "clocks": clocks4, "e2e": e2e4 if e2e4 is not None else e2e, "roofline": roof,
            "roofline_note": "`roofline` is the dominant kernel in rank 0's configs[1] pass (per-kernel events); `roofline_whole_direction` is THIS job",
            "roofline_whole_direction": whole_direction(nb, clen4, c_ms, d_ms, world),
            "cpu_baseline": cpu_baseline_block(sample, ncores, C4_LEVEL, True, f"the first {sample.size >> 30} GiB of the workload")}
    print(json.dumps(line), flush=True)
    dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what this project's codec computed: it needs --impl ours")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    ncores = os.cpu_count() or 1
    if args.impl == "reference":
        return main_reference(args, rank, world, ncores)
    try:
        return main_ours(args, rank, world, local, ncores)
    except BaseException:
        # under torchrun a rank that raises must take the job down NOW: its peers sit in exchanges only it can complete
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        if world > 1:
            os._exit(1)
        raise


if __name__ == "__main__":
    sys.exit(main())

"""Patch-mode benchmark: a 1 GiB OLD and a 1 GiB NEW (OLD rotated by half, with edits and a moved range -- tests/test_patch_ldm.py
patch_pair), 2 MiB frames, level 3, checksum on, window log ilog2(len(OLD)) + 1.  Reports, from one run on the GPU:
  * the index build of long-distance matching: a prefix call on a 4 KiB NEW with LDM on, minus the same call with LDM off;
  * compress with LDM against the same prefix call without it, and decompress with the prefix (host-pointer calls, host clock around
    a call that ends in a device synchronise; both include uploading the 1 GiB prefix and the pipeline's copies);
  * the patch size, and against libzstd's patch over the first frames (level 3, the same window log, LDM on);
  * the card's name and power limit, read in the same run.
libzstd rereads the whole prefix for every frame, so its patch is measured on the first --ref-frames frames.
The result is printed as JSON and, with --out, also written to that file.
usage: python tools/patch_bench.py [--size-mib 1024] [--reps 3] [--ref-frames 8] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size-mib", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ref-frames", type=int, default=8)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    ns = ap.parse_args()
    log = lambda *a: print(*a, flush=True)                                              # noqa: E731
    import torch
    assert torch.cuda.is_available(), "patch_bench measures the GPU codec: no CUDA device"
    import zeekstd_b200 as zk
    from zeekstd_b200 import corpus
    import test_patch_ldm as T

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    n = ns.size_mib << 20
    log("card:", card)
    old = corpus.make_mix(n, seed=7).numpy()
    new = T.patch_pair(old, seed=13, edits=64, moved=1 << 20)
    wl = T.patch_window_log(old.size)
    ctx = zk.Context(0)
    fs, lvl = 2 << 20, 3

    def timed(fn):
        ts = []
        for _ in range(ns.reps):
            torch.cuda.synchronize(); t = time.perf_counter(); r = fn(); ts.append(time.perf_counter() - t)
        return float(np.median(ts)), r

    def with_ldm(on, fn):
        ctx.set_cparameter(zk.CParameter.WindowLog(wl if on else 0)).set_cparameter(zk.CParameter.EnableLongDistanceMatching(on))
        try:
            return fn()
        finally:
            ctx.set_cparameter(zk.CParameter.WindowLog(0)).set_cparameter(zk.CParameter.EnableLongDistanceMatching(False))

    tiny = new[: 4096]
    run_tiny = lambda: ctx.compress_frames(tiny, fs, lvl, True, prefix=old)            # noqa: E731
    run_big = lambda: ctx.compress_frames(new, fs, lvl, True, prefix=old)              # noqa: E731
    log("inputs ready"); with_ldm(True, run_tiny); with_ldm(False, run_tiny)                                 # warm-up (allocations, modules)
    t_tiny_ldm, _ = with_ldm(True, lambda: timed(run_tiny))
    t_tiny, _ = with_ldm(False, lambda: timed(run_tiny))
    t_ldm, (comp, cs, ds) = with_ldm(True, lambda: timed(run_big))
    log("compress ldm", t_ldm)
    t_plain, (comp0, _, _) = with_ldm(False, lambda: timed(run_big))
    log("compress no ldm", t_plain)
    co = np.concatenate([[0], np.cumsum(cs)]).astype(np.uint64); do = np.concatenate([[0], np.cumsum(ds)]).astype(np.uint64)
    ctx.set_dparameter(zk.DParameter.WindowLogMax(wl))
    buf = np.concatenate([comp, np.zeros(64, np.uint8)])
    t_dec, (out, st, rc) = timed(lambda: ctx.decompress_frames(buf, co, do, True, prefix=old))
    assert rc == 0 and out.tobytes() == new.tobytes()
    log("decompress", t_dec)
    # libzstd references (and indexes) the whole prefix again for every frame, about a second each at 1 GiB: compare the first
    # `--ref-frames` frames only
    nref = min(ns.ref_frames, len(cs))
    t = time.perf_counter()
    ref = []
    for k in range(nref):
        ref += T.zstd_compress(new[k * fs: (k + 1) * fs], fs, lvl, prefix=old, window_log=wl, ldm=True)[0]
        log("libzstd frame", k, len(ref[-1]), int(cs[k]))
    t_ref = time.perf_counter() - t
    ref_size = sum(len(f) for f in ref); ours_size = int(np.sum(cs[:nref]))
    res = {
        "card": card, "torch_device": torch.cuda.get_device_name(0),
        "workload": {"old_bytes": int(old.size), "new_bytes": int(new.size), "frame_size": fs, "level": lvl, "window_log": wl, "checksum": True},
        "timing": "host clock around synchronous host-pointer calls (each ends in a device synchronise), median of %d; includes the 1 GiB prefix upload" % ns.reps,
        "index_build_s": t_tiny_ldm - t_tiny, "prefix_call_4KiB_s": {"ldm": t_tiny_ldm, "no_ldm": t_tiny},
        "compress_s": {"ldm": t_ldm, "no_ldm": t_plain, "ldm_over_no_ldm": t_ldm / t_plain},
        "compress_GBps_of_new": {"ldm": new.size / t_ldm / 1e9, "no_ldm": new.size / t_plain / 1e9},
        "decompress_prefix_s": t_dec, "decompress_GBps": new.size / t_dec / 1e9,
        "patch_bytes": {"ldm": int(comp.size), "no_ldm": int(comp0.size), "ldm_pct_of_new": 100.0 * comp.size / new.size,
                        "no_ldm_pct_of_new": 100.0 * comp0.size / new.size},
        "vs_libzstd_first_frames": {"frames": nref, "ours_ldm": ours_size, "libzstd_l3_ldm": ref_size, "ours_over_libzstd": ours_size / ref_size,
                                    "libzstd_single_thread_s": t_ref},
    }
    if ns.out:
        os.makedirs(os.path.dirname(os.path.abspath(ns.out)), exist_ok=True)
        json.dump(res, open(ns.out, "w"), indent=1)
    log(json.dumps(res, indent=1))
    ctx.close()


if __name__ == "__main__":
    main()

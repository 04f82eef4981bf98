"""Rate and ratio of the three DEFLATE levels on the c5 corpus, against zlib on the host.

The corpus is bench.py's c5 workload: 16,384 entries of 256 KiB sliced from synth.TextPool(64 MiB, seed 5) at
pool.offsets(), 4 GiB in all.  One job per level (fast = OTZ_M_FAST, default, best = OTZ_M_BEST) runs through the
otz_deflate_* seam on a device-resident input, the levels alternating round by round; a rate is the source bytes over the
device time (CUDA events) of one otz_deflate_run.  Then:
  - the ratio of each level (source bytes over the dense arena);
  - zlib level 6 and 9 on the same sources as whole entries (raw DEFLATE), all host cores;
  - zlib level 9's throughput on all host cores (one thread per core; zlib releases the GIL) over every 16th entry;
  - every best-level stream decoded with zlib and compared with its source, every CRC with zlib.crc32;
  - SHA-256 of each level's dense arena (comparable between builds: OTEZIP_B200_LIB selects another one);
  - the card's name and power limit, read in the same run.

  python tools/deflate_best_bench.py [--entries N] [--rounds R] [--levels fast,default,best] [--out FILE]
"""
import argparse
import concurrent.futures as cf
import hashlib
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

LEVELS = {"fast": 8 | 0x100, "default": 8, "best": 8 | 0x200}
SIZE = 262144


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=60)
        name, pl = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return name, pl
    except Exception as e:   # the numbers are still device-timed; say that the card was not identified
        return "unknown (%s)" % type(e).__name__, "unknown"


def zraw(s, level):
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    return len(c.compress(s) + c.flush())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=int, default=16384)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--levels", default="fast,default,best")
    ap.add_argument("--no-zlib", action="store_true", help="skip the host zlib numbers")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from otezip_b200 import Ctx, synth
    levels = a.levels.split(",")
    n = a.entries
    pool = synth.TextPool(64 << 20, seed=5)
    offs = pool.offsets([SIZE] * n)
    ctx = Ctx(0)
    img = ctx.pinned(n * SIZE)
    srcs = []
    for i in range(n):
        d = pool.at(offs[i], SIZE)
        img[i * SIZE:(i + 1) * SIZE] = np.frombuffer(d, dtype=np.uint8)
        srcs.append(d)
    d_in = ctx.dev_alloc(img.nbytes)
    ctx.h2d(d_in, img)
    in_ofs = np.arange(n, dtype=np.uint64) * SIZE
    in_len = np.full(n, SIZE, dtype=np.uint32)
    jobs = {lv: ctx.deflate_plan(in_ofs, in_len, np.full(n, LEVELS[lv], dtype=np.uint16)) for lv in levels}
    ctx.sync()
    for lv in levels:   # warm-up: module load, first touch of every buffer
        ctx.deflate_run(jobs[lv], d_in, img.nbytes)
    ctx.sync()
    ms = {lv: [] for lv in levels}
    for _ in range(a.rounds):
        for lv in levels:
            ctx.timer_start()
            ctx.deflate_run(jobs[lv], d_in, img.nbytes)
            ms[lv].append(ctx.timer_stop())
    name, pl = card()
    res = {"gpu": name, "power_limit": pl, "entries": n, "entry_bytes": SIZE, "source_bytes": n * SIZE,
           "corpus": "bench.py c5: synth.TextPool(64 MiB, seed 5), pool.offsets([262144] * entries)", "rounds": a.rounds,
           "levels": {}}
    tot_in = n * SIZE
    best_ok = None
    for lv in levels:
        o, sz, crc, mo, total = ctx.deflate_results(jobs[lv], n)
        out = ctx.deflate_fetch(jobs[lv], total)
        med = float(np.median(ms[lv]))
        res["levels"][lv] = {"ms": [round(x, 3) for x in ms[lv]], "GB_per_s": round(tot_in / med / 1e6, 2), "ratio": round(tot_in / total, 4),
                             "compressed_bytes": int(total), "stored_entries": int((mo == 0).sum()),
                             "sha256_dense": hashlib.sha256(out.tobytes()).hexdigest()}
        if lv == "best":
            def chk(i):
                p = out[int(o[i]):int(o[i]) + int(sz[i])].tobytes()
                dec = zlib.decompress(p, -15) if mo[i] == 8 else p
                return dec == srcs[i] and int(crc[i]) == (zlib.crc32(srcs[i]) & 0xFFFFFFFF)
            with cf.ThreadPoolExecutor(os.cpu_count()) as ex:
                best_ok = sum(ex.map(chk, range(n)))
            res["levels"][lv]["streams_verified"] = "%d / %d decoded by zlib to their source, CRC-32 equal" % (best_ok, n)
    ctx.dev_free(d_in)
    for j in jobs.values():
        ctx.deflate_destroy(j)
    ctx.close()
    if not a.no_zlib:
        cores = os.cpu_count()
        with cf.ThreadPoolExecutor(cores) as ex:
            z6 = sum(ex.map(lambda s: zraw(s, 6), srcs))
            z9 = sum(ex.map(lambda s: zraw(s, 9), srcs))
            sample = srcs[::16]
            t0 = time.perf_counter()
            list(ex.map(lambda s: zraw(s, 9), sample))
            dt = time.perf_counter() - t0
        res["zlib"] = {"level6_whole_entries_ratio": round(tot_in / z6, 4), "level9_whole_entries_ratio": round(tot_in / z9, 4),
                       "level9_GB_per_s_all_cores": round(len(sample) * SIZE / dt / 1e9, 3), "host_cores": cores,
                       "level9_sample": "every 16th entry, %d entries" % len(sample)}
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    if best_ok is not None and best_ok != n:
        sys.exit("best-level streams that do not decode to their source: %d" % (n - best_ok))


if __name__ == "__main__":
    main()

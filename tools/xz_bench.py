"""XZ (ZIP method 95) read path on the GPU.  Prints one JSON line:

  many_gbps          --entries JSON-log entries of floor(2^U(12,22)) bytes, xz preset 6, CRC64 (single-threaded xz output: one
                     dictionary reset per entry, so one segment per entry)
  reset_gbps         the same bytes with a dictionary reset every --reset-kib KiB (default 1 MiB; raw LZMA2 pieces in one
                     block): the segment parallelism inside an entry
  single_64mib_gbps  --big entries of 64 MiB at preset 6, one segment each: the per-stream rate
  liblzma_gbps       lzma.decompress of the entries of many_* on all host cores (a thread pool; the module releases the GIL)
  gpu, power_limit   what the numbers were measured on

Every GPU rate is uncompressed bytes over device time (CUDA events around otz_extract_run on device-resident buffers, L2
flushed before every run, after --warmup runs, mean of --steps); the output of the last run is compared with the input before
it counts.  Usage: python tools/xz_bench.py [--entries N] [--steps K] [--warmup W] [--big N] [--reset-kib K]"""
import argparse
import json
import lzma
import os
import random
import sys
import time
from concurrent.futures import ThreadPoolExecutor

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from otezip_b200 import synth  # noqa: E402
from tests.test_xz_cpu import raw_lzma2, stream  # noqa: E402
from tools.deflate64_bench import card, timed, zip_image  # noqa: E402


def reset_every(r: bytes, step: int) -> bytes:
    pieces = [r[o:o + step] for o in range(0, len(r), step)] or [b""]
    raw = b"".join(raw_lzma2(p, preset=6)[:-1] for p in pieces) + b"\x00"
    return stream([(raw, r, {})], check=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--big", type=int, default=3, help="64 MiB entries of the single-stream measurement")
    ap.add_argument("--reset-kib", type=int, default=1024, help="dictionary reset interval of the reset_* corpus")
    a = ap.parse_args()
    name, limit = card()
    rnd = random.Random(7)
    pool = synth.TextPool(32 << 20, 7)
    raws = [pool.take(int(2 ** rnd.uniform(12, 22))) for _ in range(a.entries)]
    bigs = [pool.take(64 << 20) for _ in range(a.big)]
    with ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        many = list(ex.map(lambda r: lzma.compress(r, preset=6, check=lzma.CHECK_CRC64), raws))
        reset = list(ex.map(lambda r: reset_every(r, a.reset_kib << 10), raws))
        big = list(ex.map(lambda r: lzma.compress(r, preset=6, check=lzma.CHECK_CRC64), bigs))
    out_bytes = sum(len(r) for r in raws)
    res = {"tool": "xz_bench", "gpu": name, "power_limit": limit, "entries": a.entries, "out_bytes": out_bytes,
           "reset_kib": a.reset_kib, "many_comp_bytes": sum(map(len, many)), "reset_comp_bytes": sum(map(len, reset))}
    for rep in range(2):
        for key, pay in (("many", many), ("reset", reset)):
            g, ms = timed(zip_image(95, pay, raws), raws, a.steps, a.warmup)
            res.setdefault(key + "_gbps", []).append(round(g, 2))
            res.setdefault(key + "_ms", []).append(round(ms, 3))
    if a.big:
        g, ms = timed(zip_image(95, big, bigs), bigs, max(1, a.steps // 2), 1)
        res["single_64mib_entries"], res["single_64mib_gbps"], res["single_64mib_ms"] = a.big, round(g, 3), round(ms, 2)
    cores = os.cpu_count() or 1
    with ThreadPoolExecutor(cores) as ex:
        t = time.perf_counter()
        dec = list(ex.map(lzma.decompress, many))
        dt = time.perf_counter() - t
    assert dec == raws
    res["liblzma_cores"], res["liblzma_gbps"] = cores, round(out_bytes / dt / 1e9, 3)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

"""Deflate64 (ZIP method 9) read path on the GPU.  Prints one JSON line:

  dual_*_gbps        one corpus of "dual" streams (32 KiB window, matches <= 257 bytes: the same bytes mean the same thing as
                     DEFLATE and as Deflate64), decoded as method 8 under OTZ_INFLATE_MODE=legacy (k_inflate, DEFLATE tables),
                     as method 9 (k_inflate<G, W, true>) and as method 8 on the default two-phase path
  dual_ratio         method-9 GB/s over legacy method-8 GB/s on identical bytes: the cost of the Deflate64 variant
  native_gbps        native Deflate64 streams of the same data (64 KiB window, matches up to 65,538 bytes)
  single_64mib_gbps  a handful of 64 MiB native entries, one tile each (the single-stream rate of a large file)
  gpu, power_limit   what the numbers were measured on

Corpus: seeded JSON-log text (otezip_b200.synth), --entries entries of floor(2^U(12,22)) bytes, encoded by tools/d64enc.c on
all host cores.  Every rate is uncompressed bytes over device time (CUDA events around otz_extract_run on device-resident
buffers, after --warmup runs, mean of --steps); the output of the last run is compared with the input before it counts.
Usage: python tools/deflate64_bench.py [--entries N] [--steps K] [--warmup W] [--big N]"""
import argparse
import json
import os
import random
import struct
import subprocess
import sys
import zlib
from concurrent.futures import ThreadPoolExecutor

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from otezip_b200 import Ctx, synth  # noqa: E402
from otezip_b200.native import parse_central, default_opts  # noqa: E402
from tests.deflate64 import Encoder  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, limit = [x.strip() for x in r.stdout.splitlines()[0].split(",")]
        return name, limit
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def zip_image(method, payloads, raws):
    out, cd = bytearray(), bytearray()
    for k, (p, r) in enumerate(zip(payloads, raws)):
        name, crc = b"e%05d" % k, zlib.crc32(r)
        ofs = len(out)
        out += struct.pack("<IHHHHHIIIHH", 0x04034B50, 20, 0, method, 0, 0x21, crc, len(p), len(r), len(name), 0) + name + p
        cd += struct.pack("<IHHHHHHIIIHHHHHII", 0x02014B50, 0x031E, 20, 0, method, 0, 0x21, crc, len(p), len(r), len(name), 0, 0, 0, 0,
                          0o100644 << 16, ofs) + name
    n = len(payloads)
    return bytes(out + cd + struct.pack("<IHHHHIIH", 0x06054B50, 0, 0, n, n, len(cd), len(out), 0))


def timed(img, raws, steps, warmup, env=None):
    """-> GB/s of otz_extract_run over the image (device time), after checking the decoded bytes"""
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        c = Ctx(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v
    tab = parse_central(img)
    out_len = int((tab["out_ofs"].astype(np.int64) + tab["uncomp_size"]).max())
    h = c.pinned(len(img))
    h[:] = np.frombuffer(img, np.uint8)
    d_arch, d_out = c.dev_alloc(len(img)), c.dev_alloc(out_len)
    c.h2d(d_arch, h)
    plan = c.plan(tab, default_opts())
    for _ in range(warmup):
        c.run(plan, d_arch, len(img), d_out, out_len)
    ms = []
    for _ in range(steps):
        c.flush_l2()
        c.timer_start()
        c.run(plan, d_arch, len(img), d_out, out_len)
        ms.append(c.timer_stop())
    crc, st = c.results(plan, len(tab))
    got = c.pinned(out_len)
    c.d2h(got, d_out)
    c.sync()
    for k, r in enumerate(raws):
        o = int(tab["out_ofs"][k])
        assert int(st[k]) & 0xFF == 0 and int(crc[k]) == zlib.crc32(r) and got[o:o + len(r)].tobytes() == r, (k, hex(int(st[k])))
    c.plan_destroy(plan)
    c.dev_free(d_arch)
    c.dev_free(d_out)
    c.pinned_free(h)
    c.pinned_free(got)
    c.close()
    total = sum(len(r) for r in raws)
    return total / (sum(ms) / len(ms) * 1e-3) / 1e9, sum(ms) / len(ms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--big", type=int, default=4, help="64 MiB native entries of the single-stream measurement")
    a = ap.parse_args()
    name, limit = card()
    rnd = random.Random(7)
    pool = synth.TextPool(32 << 20, 7)
    raws = [pool.take(int(2 ** rnd.uniform(12, 22))) for _ in range(a.entries)]
    enc = Encoder()
    with ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        dual = list(ex.map(lambda r: enc.compress(r, "dual"), raws))
        native = list(ex.map(lambda r: enc.compress(r, "deflate64"), raws))
        bigs = [pool.take(64 << 20) for _ in range(a.big)]
        big_native = list(ex.map(lambda r: enc.compress(r, "deflate64"), bigs))
    res = {"tool": "deflate64_bench", "gpu": name, "power_limit": limit, "entries": a.entries,
           "out_bytes": sum(len(r) for r in raws), "dual_comp_bytes": sum(map(len, dual)), "native_comp_bytes": sum(map(len, native))}
    legacy = {"OTZ_INFLATE_MODE": "legacy"}
    # the three dual runs alternate twice, so that drift of the shared machine shows as spread
    for rep in range(2):
        for key, m, env in (("dual_m8_legacy", 8, legacy), ("dual_m9", 9, None), ("dual_m8_default", 8, None)):
            g, ms = timed(zip_image(m, dual, raws), raws, a.steps, a.warmup, env)
            res.setdefault(key + "_gbps", []).append(round(g, 2))
            res.setdefault(key + "_ms", []).append(round(ms, 3))
    res["dual_ratio"] = round(sum(res["dual_m9_gbps"]) / sum(res["dual_m8_legacy_gbps"]), 3)
    g, ms = timed(zip_image(9, native, raws), raws, a.steps, a.warmup)
    res["native_gbps"], res["native_ms"] = round(g, 2), round(ms, 3)
    if a.big:
        g, ms = timed(zip_image(9, big_native, bigs), bigs, max(1, a.steps // 2), 1)
        res["single_64mib_entries"], res["single_64mib_gbps"], res["single_64mib_ms"] = a.big, round(g, 3), round(ms, 2)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

"""WinZip AES read path on the GPU: the configs[2] archive (bench.py workload "c3"), its payloads sealed as AES-256 AE-2 by
otz_aes_seal, then decrypted and decoded on the device.  Prints one JSON line:

  plain_gbps / aes_gbps     device-timed decode of the plain archive, and decrypt + decode of the sealed one (key derivation,
                            CTR, authentication codes, decode, verdicts), uncompressed bytes per second, same process
  split_ms                  KDF / CTR / MAC (side stream, from the end of the KDF) / decode of the plaintext image, device events
  mac_largest_ms            the authentication code of the largest entry alone (one serial HMAC-SHA1 chain)
  e2e_*_s                   zip_open + zip_fopen_index of every entry + zip_close, plain and encrypted archive files of the
                            first --e2e-entries entries
  cpu_kdf_s                 hashlib.pbkdf2_hmac for the same number of salts on all cores (the CPU comparison)
  gpu, power_limit          what the numbers were measured on

Before timing, 1 % of the sealed entries are opened by tests/aeszip.py (an independent implementation) and compared.
Usage: python tools/aes_bench.py [--entries N] [--steps K] [--warmup W] [--out FILE]"""
import argparse
import json
import multiprocessing as mp
import os
import struct
import subprocess
import sys
import tempfile
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

PW = b"aes-bench password"


def _kdf(salt):
    import hashlib
    return hashlib.pbkdf2_hmac("sha1", PW, salt, 1000, 66)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, limit = [x.strip() for x in r.stdout.splitlines()[0].split(",")]
        return name, limit
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def zip_image(names, payloads, tab, method, flags, extra):
    """ZIP32 image of the given payloads (method / flags / extra field per entry)."""
    out, cd = bytearray(), bytearray()
    for k, (name, pay) in enumerate(zip(names, payloads)):
        crc, un = int(tab["crc32"][k]), int(tab["uncomp_size"][k])
        crc = 0 if method == 99 else crc
        ofs = len(out)
        out += struct.pack("<IHHHHHIIIHH", 0x04034B50, 20, flags, method, 0, 0x21, crc, len(pay), un, len(name), len(extra)) + name + extra + pay
        cd += struct.pack("<IHHHHHHIIIHHHHHII", 0x02014B50, 0x031E, 20, flags, method, 0, 0x21, crc, len(pay), un, len(name), len(extra),
                          0, 0, 0, 0o100644 << 16, ofs) + name + extra
    n = len(payloads)
    return bytes(out + cd + struct.pack("<IHHHHIIH", 0x06054B50, 0, 0, n, n, len(cd), len(out), 0))


def e2e(path, pw):
    from otezip_b200.zipapi import ZipApi
    api = ZipApi()
    t0 = time.perf_counter()
    za = api.L.zip_open(path.encode(), 0, None)
    if pw:
        api.L.zip_set_default_password(za, pw)
    ok = 0
    for i in range(api.L.zip_get_num_files(za)):
        zf = api.L.zip_fopen_index(za, i, 0)
        ok += bool(zf)
        if zf:
            api.L.zip_fclose(zf)
    api.L.zip_close(za)
    return time.perf_counter() - t0, ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=int, default=10000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--e2e-entries", type=int, default=1000, help="entries of the archive files of the end-to-end leg")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bench
    from otezip_b200 import Ctx
    from otezip_b200.native import AES_ENTRY_DTYPE, default_opts
    from tests import aeszip

    ctx = Ctx(0)
    wl = bench.workload("c3", 0, 1, args.entries, ctx.pinned)
    img, tab = wl["image"], wl["table"]
    n = len(tab)
    un_bytes = int(tab["uncomp_size"].astype(np.int64).sum())
    hb = img.tobytes()
    data_ofs = np.array([int(t) + 30 + struct.unpack_from("<H", hb, int(t) + 26)[0] + struct.unpack_from("<H", hb, int(t) + 28)[0]
                         for t in tab["lfh_ofs"]], dtype=np.uint64)
    comp = tab["comp_size"].astype(np.uint64)
    # sealed layout (each ciphertext 16-byte aligned) and plaintext-image layout (each payload 16-byte aligned)
    pre = 16 + 2
    seal_rows = np.zeros(n, dtype=AES_ENTRY_DTYPE)
    open_rows = np.zeros(n, dtype=AES_ENTRY_DTYPE)
    s_pos = p_pos = 0
    for k in range(n):
        s = ((s_pos + pre + 15) & ~15) - pre
        p = ((p_pos + 30 + 15) & ~15) - 30
        seal_rows[k] = (s, int(data_ofs[k]), int(comp[k]), 3, 0)
        open_rows[k] = (s, p, int(comp[k]) + 28, 3, 0)
        s_pos = s + int(comp[k]) + 28
        p_pos = p + 30 + int(comp[k])
    d_img = ctx.dev_alloc(img.nbytes)
    ctx.h2d(d_img, img)
    d_sealed = ctx.dev_alloc(s_pos)
    d_plain = ctx.dev_alloc(p_pos)
    d_out = ctx.dev_alloc(wl["out_bytes"])
    salts = os.urandom(16 * n)
    ctx.aes_seal(d_img, img.nbytes, seal_rows, salts, [PW], d_sealed, s_pos)
    sealed = np.zeros(s_pos, dtype=np.uint8)
    ctx.d2h(sealed, d_sealed)
    ctx.sync()
    sb = sealed.tobytes()
    rng = np.random.default_rng(7)
    check = sorted(rng.choice(n, max(1, n // 100), replace=False).tolist())
    for k in check:
        o, sz = int(seal_rows["payload_ofs"][k]), int(comp[k]) + 28
        assert sb[o:o + 16] == salts[16 * k:16 * k + 16]
        want = hb[int(data_ofs[k]):int(data_ofs[k]) + int(comp[k])]
        assert aeszip.open_payload(sb[o:o + sz], PW, 3) == want, k

    inner = tab.copy()
    inner["lfh_ofs"] = open_rows["data_ofs"]
    plan_plain = ctx.plan(tab, default_opts())
    plan_aes = ctx.plan(inner, default_opts())
    ctx.sync()

    def plain_step():
        ctx.run(plan_plain, d_img, img.nbytes, d_out, wl["out_bytes"])

    def aes_step():
        ctx.aes_open(d_sealed, s_pos, open_rows, [PW], d_plain, p_pos)
        ctx.run(plan_aes, d_plain, p_pos, d_out, wl["out_bytes"])
        return ctx.aes_status(n)

    for _ in range(args.warmup):
        plain_step()
        aes_step()
    ctx.sync()
    crc, st = ctx.results(plan_aes, n)
    verdict = aes_step()
    crc, st = ctx.results(plan_aes, n)
    if np.count_nonzero(verdict) or np.count_nonzero(st) or not np.array_equal(crc, tab["crc32"]):
        raise SystemExit("aes_bench: %d verdicts / %d statuses not OK — numbers would be invalid" % (np.count_nonzero(verdict), np.count_nonzero(st)))
    res = {"entries": n, "uncomp_bytes": un_bytes, "comp_bytes": int(comp.sum()), "steps": args.steps, "spot_checked": len(check)}
    # plain and AES alternating, each timed over `steps` steps
    pl, ae = [], []
    for _ in range(2):
        ctx.sync()
        ctx.timer_start()
        for _ in range(args.steps):
            plain_step()
        pl.append(ctx.timer_stop())
        ctx.sync()
        ctx.timer_start()
        for _ in range(args.steps):
            aes_step()
        ae.append(ctx.timer_stop())
    res["plain_ms_per_step"] = [round(x / args.steps, 3) for x in pl]
    res["aes_ms_per_step"] = [round(x / args.steps, 3) for x in ae]
    res["plain_gbps"] = round(un_bytes * args.steps / (min(pl) / 1e3) / 1e9, 2)
    res["aes_gbps"] = round(un_bytes * args.steps / (min(ae) / 1e3) / 1e9, 2)
    # split of one AES step: KDF / CTR / MAC from the seam's events, decode of the plaintext image on its own
    aes_step()
    kdf, ctr, mac = ctx.aes_times()
    ctx.sync()
    ctx.timer_start()
    ctx.run(plan_aes, d_plain, p_pos, d_out, wl["out_bytes"])
    dec = ctx.timer_stop()
    res["split_ms"] = {"kdf": round(kdf, 3), "ctr": round(ctr, 3), "mac_from_kdf_end": round(mac, 3), "decode": round(dec, 3)}
    big = int(np.argmax(comp))
    ctx.aes_open(d_sealed, s_pos, open_rows[big:big + 1], [PW], d_plain, p_pos)
    assert ctx.aes_status(1)[0] == 0
    res["mac_largest_ms"] = round(ctx.aes_times()[2], 3)
    res["largest_entry_comp_bytes"] = int(comp[big])
    # end to end through the libzip API
    m = min(n, args.e2e_entries)
    names = [b"e/%05d.bin" % k for k in range(m)]
    plains = [hb[int(data_ofs[k]):int(data_ofs[k]) + int(comp[k])] for k in range(m)]
    encs = [sb[int(seal_rows["payload_ofs"][k]):int(seal_rows["payload_ofs"][k]) + int(comp[k]) + 28] for k in range(m)]
    tmp = tempfile.mkdtemp()
    pp, pe = os.path.join(tmp, "plain.zip"), os.path.join(tmp, "aes.zip")
    open(pp, "wb").write(zip_image(names, plains, tab, 8, 0, b""))
    open(pe, "wb").write(zip_image(names, encs, tab, 99, 1, struct.pack("<HHH2sBH", 0x9901, 7, 2, b"AE", 3, 8)))
    del plains, encs
    tp, okp = e2e(pp, None)
    te, oke = e2e(pe, PW)
    os.unlink(pp)
    os.unlink(pe)
    res.update(e2e_entries=m, e2e_uncomp_bytes=int(tab["uncomp_size"][:m].astype(np.int64).sum()), e2e_plain_s=round(tp, 3), e2e_aes_s=round(te, 3),
               e2e_entries_ok=[okp, oke])
    # CPU comparison: the same number of PBKDF2 runs (AES-256: 66 bytes, 4 output blocks) on every core
    salt_list = [salts[16 * k:16 * k + 16] for k in range(n)]
    t0 = time.perf_counter()
    with mp.Pool(os.cpu_count()) as pool:
        pool.map(_kdf, salt_list, chunksize=64)
    res["cpu_kdf_s"] = round(time.perf_counter() - t0, 3)
    res["cpu_cores"] = os.cpu_count()
    res["gpu"], res["power_limit"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    for p in (plan_plain, plan_aes):
        ctx.plan_destroy(p)
    for d in (d_img, d_sealed, d_plain, d_out):
        ctx.dev_free(d)
    ctx.close()


if __name__ == "__main__":
    main()

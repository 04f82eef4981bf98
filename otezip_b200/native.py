"""ctypes loader for libotezip_b200.so (include/otz_gpu.h).  Fails loudly when the library is
missing; there is no fallback."""
from __future__ import annotations

import ctypes as C
import os
import struct

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def lib_path() -> str:
    """OTEZIP_B200_LIB selects another build of the same library (the bounds-checked one, libotezip_b200_dbg.so)."""
    return os.environ.get("OTEZIP_B200_LIB") or os.path.join(HERE, "libotezip_b200.so")


class OtzEntry(C.Structure):  # struct otz_entry, include/otz_gpu.h
    _fields_ = [("lfh_ofs", C.c_uint64), ("out_ofs", C.c_uint64), ("comp_size", C.c_uint32),
                ("uncomp_size", C.c_uint32), ("crc32", C.c_uint32), ("method", C.c_uint16), ("flags", C.c_uint16)]


ENTRY_DTYPE = np.dtype([("lfh_ofs", "<u8"), ("out_ofs", "<u8"), ("comp_size", "<u4"), ("uncomp_size", "<u4"),
                        ("crc32", "<u4"), ("method", "<u2"), ("flags", "<u2")])
assert ENTRY_DTYPE.itemsize == C.sizeof(OtzEntry) == 32


class OtzOpts(C.Structure):  # struct otz_extract_opts
    _fields_ = [("ignore_zipbomb", C.c_int), ("max_ratio", C.c_uint64), ("max_slack", C.c_uint64),
                ("verify_only", C.c_int)]


def default_opts(verify_only: int = 0, ignore_zipbomb: int = 0) -> OtzOpts:
    return OtzOpts(ignore_zipbomb, 1000, 1 << 20, verify_only)


ST_OK = 0
STF_CRC_MISMATCH, STF_REF_EOB, STF_SHORT = 0x100, 0x200, 0x400


class OtzAesEntry(C.Structure):  # struct otz_aes_entry
    _fields_ = [("payload_ofs", C.c_uint64), ("data_ofs", C.c_uint64), ("size", C.c_uint32), ("strength", C.c_uint16),
                ("password", C.c_uint16)]


AES_ENTRY_DTYPE = np.dtype([("payload_ofs", "<u8"), ("data_ofs", "<u8"), ("size", "<u4"), ("strength", "<u2"), ("password", "<u2")])
assert AES_ENTRY_DTYPE.itemsize == C.sizeof(OtzAesEntry) == 24
ST_NOPASSWD, ST_WRONGPASSWD, ST_AUTH = 11, 12, 13


class Lib:
    _inst = None

    def __init__(self):
        p = lib_path()
        if not os.path.exists(p):
            raise RuntimeError("libotezip_b200.so is not built (run `make` or __graft_entry__.build()); "
                               "there is no CPU fallback")
        L = self.L = C.CDLL(p)
        vp, u64, u32p, i32p = C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_int32)
        L.otz_last_error.restype = C.c_char_p
        L.otz_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
        L.otz_ctx_destroy.argtypes = [vp]
        L.otz_ctx_destroy.restype = None
        L.otz_sm_count.argtypes = [vp]
        L.otz_pci_bus_id.argtypes = [vp, C.c_char_p, C.c_int]
        L.otz_launch_count.argtypes = [vp]
        L.otz_launch_count.restype = u64
        L.otz_dev_alloc.argtypes = [vp, u64, C.POINTER(vp)]
        L.otz_dev_free.argtypes = [vp, vp]
        L.otz_host_alloc.argtypes = [u64, C.POINTER(vp)]
        L.otz_host_free.argtypes = [vp]
        L.otz_h2d.argtypes = [vp, vp, vp, u64]
        L.otz_d2h.argtypes = [vp, vp, vp, u64]
        L.otz_dev_memset.argtypes = [vp, vp, C.c_int, u64]
        L.otz_sync.argtypes = [vp]
        L.otz_timer_start.argtypes = [vp]
        L.otz_timer_stop.argtypes = [vp, C.POINTER(C.c_float)]
        L.otz_profile_enable.argtypes = [vp, C.c_int]
        L.otz_profile_get.argtypes = [vp, C.c_int] + [C.POINTER(C.c_float)] * 4
        L.otz_profile_runs.argtypes = [vp]
        L.otz_flush_l2.argtypes = [vp]
        L.otz_plan_create.argtypes = [vp, vp, C.c_uint32, C.POINTER(OtzOpts), C.POINTER(vp)]
        L.otz_plan_destroy.argtypes = [vp, vp]
        L.otz_plan_destroy.restype = None
        L.otz_extract_run.argtypes = [vp, vp, vp, u64, vp, u64]
        L.otz_extract_results.argtypes = [vp, vp, vp, vp]
        L.otz_extract_host.argtypes = [vp, vp, u64, vp, C.c_uint32, C.POINTER(OtzOpts), vp, u64, vp, vp]
        L.otz_status_accepts.argtypes = [C.c_int32, C.c_int, C.c_int]
        L.otz_partition.argtypes = [vp, C.c_uint32, C.c_uint32, vp]
        L.otz_inflate_fallbacks.argtypes = [vp]
        L.otz_inflate_fallbacks.restype = C.c_uint32
        L.otz_deflate_plan.argtypes = [vp, vp, vp, vp, C.c_uint32, C.POINTER(vp)]
        L.otz_deflate_destroy.argtypes = [vp, vp]
        L.otz_deflate_destroy.restype = None
        L.otz_deflate_run.argtypes = [vp, vp, vp, u64]
        L.otz_deflate_results.argtypes = [vp, vp, vp, vp, vp, vp, C.POINTER(u64)]
        L.otz_deflate_device_output.argtypes = [vp]
        L.otz_deflate_device_output.restype = vp
        L.otz_deflate_fetch.argtypes = [vp, vp, vp, u64]
        L.otz_deflate_chunks.argtypes = [vp, vp, vp, vp, vp, C.c_uint32, C.POINTER(C.c_uint32)]
        L.otz_deflate_host.argtypes = [vp, vp, u64, vp, vp, vp, C.c_uint32, vp, u64, vp, vp, vp, vp, C.POINTER(u64)]
        L.otz_aes_open.argtypes = [vp, vp, u64, vp, C.c_uint32, vp, C.c_uint32, vp, u64]
        L.otz_aes_status.argtypes = [vp, vp]
        L.otz_aes_times.argtypes = [vp] + [C.POINTER(C.c_float)] * 3
        L.otz_aes_seal.argtypes = [vp, vp, u64, vp, C.c_uint32, vp, vp, C.c_uint32, vp, u64]

    @classmethod
    def get(cls) -> "Lib":
        if cls._inst is None:
            cls._inst = Lib()
        return cls._inst

    def check(self, rc: int, what: str = ""):
        if rc != 0:
            raise RuntimeError("%s failed (%d): %s" % (what, rc, self.L.otz_last_error().decode()))


EF_PARENT, EF_CHUNK, EF_LAST_CHUNK = 1, 2, 4


def partition(table: np.ndarray, parts: int) -> np.ndarray:
    """otz_partition: contiguous index ranges balanced by comp + uncomp bytes -> first[parts + 1]."""
    t = np.ascontiguousarray(table)
    first = np.zeros(parts + 1, dtype=np.uint32)
    lib = Lib.get()
    lib.check(lib.L.otz_partition(t.ctypes.data_as(C.c_void_p), len(t), parts, first.ctypes.data_as(C.c_void_p)), "otz_partition")
    return first


def expand_chunk_index(img, tab: np.ndarray) -> np.ndarray:
    """Host-side mirror of otezip.c:chunk_index_of/run_window: entries whose LFH extra field carries the 'OZ' chunk
    index become a PARENT row plus one CHUNK row per chunk (appended after the entry rows)."""
    b = memoryview(img)
    rows = []
    out = tab.copy()
    for k in range(len(tab)):
        if int(tab["method"][k]) != 8:
            continue
        lfh = int(tab["lfh_ofs"][k])
        nl, xl = struct.unpack_from("<HH", b, lfh + 26)
        x = bytes(b[lfh + 30 + nl:lfh + 30 + nl + xl])
        o = 0
        while o + 4 <= len(x):
            hid, sz = struct.unpack_from("<HH", x, o)
            if hid == 0x5A4F and sz >= 12 and x[o + 4] == 1:
                cb, nc = struct.unpack_from("<II", x, o + 8)
                cs = struct.unpack_from("<%dI" % nc, x, o + 16)
                un = int(tab["uncomp_size"][k])
                if nc >= 2 and nc == -(-un // cb) and sum(cs) == int(tab["comp_size"][k]):
                    out["flags"][k] = EF_PARENT
                    cofs, uofs = lfh + 30 + nl + xl, 0
                    for c in range(nc):
                        u = min(cb, un - uofs)
                        rows.append((cofs, int(tab["out_ofs"][k]) + uofs, cs[c], u, k, 8,
                                     EF_CHUNK | (EF_LAST_CHUNK if c + 1 == nc else 0)))
                        cofs += cs[c]
                        uofs += u
                break
            o += 4 + sz
    if not rows:
        return out
    extra = np.array(rows, dtype=ENTRY_DTYPE)
    return np.concatenate([out, extra])


def parse_central(img) -> np.ndarray:
    """Entry table (ENTRY_DTYPE, out_ofs 16-byte aligned prefix sums) from a ZIP image.  Test/bench helper
    mirroring what the C host library's central-directory walk emits; not a decoder."""
    b = memoryview(img)
    n = len(b)
    pos = -1
    lo = max(0, n - 65558)
    tail = bytes(b[lo:])
    i = len(tail) - 22
    while i >= 0:
        if tail[i:i + 4] == b"PK\x05\x06":
            ents, sz, ofs = struct.unpack_from("<HII", tail, i + 10)
            if ents == 0xFFFF or sz == 0xFFFFFFFF or ofs == 0xFFFFFFFF:   # ZIP64: locator + 64-bit record
                p = lo + i
                if p >= 20 and bytes(b[p - 20:p - 16]) == b"PK\x06\x07":
                    rpos = struct.unpack_from("<Q", b, p - 12)[0]
                    if rpos + 56 <= n and bytes(b[rpos:rpos + 4]) == b"PK\x06\x06":
                        ents, sz, ofs = struct.unpack_from("<QQQ", b, rpos + 32)
            if ofs + sz <= n and (ents == 0 or bytes(b[ofs:ofs + 4]) == b"PK\x01\x02"):
                pos = lo + i
                break
        i -= 1
    if pos < 0:
        raise ValueError("no EOCD")
    tab = np.zeros(ents, dtype=ENTRY_DTYPE)
    off = ofs
    out = 0
    for k in range(ents):
        (sig, _, _, _, method, _, _, crc, comp, uncomp, fl, xl, cl, _, _, _, lfh) = struct.unpack_from(
            "<IHHHHHHIIIHHHHHII", b, off)
        assert sig == 0x02014B50
        if comp == 0xFFFFFFFF or uncomp == 0xFFFFFFFF or lfh == 0xFFFFFFFF:   # ZIP64 extended information
            x = bytes(b[off + 46 + fl:off + 46 + fl + xl])
            o = 0
            while o + 4 <= len(x):
                hid, hsz = struct.unpack_from("<HH", x, o)
                if hid == 1:
                    q = o + 4
                    if uncomp == 0xFFFFFFFF:
                        uncomp = struct.unpack_from("<Q", x, q)[0]
                        q += 8
                    if comp == 0xFFFFFFFF:
                        comp = struct.unpack_from("<Q", x, q)[0]
                        q += 8
                    if lfh == 0xFFFFFFFF:
                        lfh = struct.unpack_from("<Q", x, q)[0]
                    break
                o += 4 + hsz
        tab[k] = (lfh, out, comp, uncomp, crc, method, 0)
        out += (uncomp + 15) & ~15
        off += 46 + fl + xl + cl
    return tab


class Ctx:
    """One device context (stream, CRC tables, scratch)."""

    def __init__(self, device: int = 0):
        self.lib = Lib.get()
        self.L = self.lib.L
        h = C.c_void_p()
        self.lib.check(self.L.otz_ctx_create(device, C.byref(h)), "otz_ctx_create")
        self.h = h

    def close(self):
        if self.h:
            self.L.otz_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- memory
    def dev_alloc(self, nbytes: int) -> C.c_void_p:
        p = C.c_void_p()
        self.lib.check(self.L.otz_dev_alloc(self.h, nbytes, C.byref(p)), "otz_dev_alloc")
        return p

    def dev_free(self, p):
        self.L.otz_dev_free(self.h, p)

    def pinned(self, nbytes: int) -> np.ndarray:
        p = C.c_void_p()
        self.lib.check(self.L.otz_host_alloc(nbytes, C.byref(p)), "otz_host_alloc")
        arr = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(nbytes, 1),))
        return arr[:nbytes]

    def pinned_free(self, arr: np.ndarray):
        """Release a buffer obtained from pinned() (the array must not be used afterwards)."""
        if arr is not None and arr.size:
            base = arr
            while isinstance(getattr(base, "base", None), np.ndarray):
                base = base.base
            self.L.otz_host_free(C.c_void_p(base.ctypes.data))

    def h2d(self, d, h: np.ndarray, nbytes: int | None = None):
        self.lib.check(self.L.otz_h2d(self.h, d, h.ctypes.data_as(C.c_void_p), h.nbytes if nbytes is None else nbytes), "h2d")

    def d2h(self, h: np.ndarray, d, nbytes: int | None = None):
        self.lib.check(self.L.otz_d2h(self.h, h.ctypes.data_as(C.c_void_p), d, h.nbytes if nbytes is None else nbytes), "d2h")

    def sync(self):
        self.lib.check(self.L.otz_sync(self.h), "otz_sync")

    def timer_start(self):
        self.lib.check(self.L.otz_timer_start(self.h), "timer_start")

    def timer_stop(self) -> float:
        ms = C.c_float()
        self.lib.check(self.L.otz_timer_stop(self.h, C.byref(ms)), "timer_stop")
        return ms.value

    def flush_l2(self):
        self.lib.check(self.L.otz_flush_l2(self.h), "flush_l2")

    def profile(self, on: int):
        self.L.otz_profile_enable(self.h, on)

    def profile_read(self):
        """-> list of (ms_resolve, ms_decode, ms_crc, ms_finalize) for the runs since profile(1)"""
        out = []
        n = self.L.otz_profile_runs(self.h)
        for i in range(max(0, n - 64), n):
            f = [C.c_float() for _ in range(4)]
            self.lib.check(self.L.otz_profile_get(self.h, i, *[C.byref(x) for x in f]), "otz_profile_get")
            out.append(tuple(x.value for x in f))
        return out

    def pci_bus_id(self) -> str:
        b = C.create_string_buffer(64)
        self.lib.check(self.L.otz_pci_bus_id(self.h, b, 64), "otz_pci_bus_id")
        return b.value.decode()

    def sm_count(self) -> int:
        return int(self.L.otz_sm_count(self.h))

    def launches(self) -> int:
        return int(self.L.otz_launch_count(self.h))

    # -- read path
    def plan(self, table: np.ndarray, opts: OtzOpts):
        p = C.c_void_p()
        t = np.ascontiguousarray(table)
        self.lib.check(self.L.otz_plan_create(self.h, t.ctypes.data_as(C.c_void_p), len(t), C.byref(opts), C.byref(p)),
                       "otz_plan_create")
        return p

    def plan_destroy(self, p):
        self.L.otz_plan_destroy(self.h, p)

    def run(self, plan, d_archive, archive_len: int, d_out, out_len: int):
        self.lib.check(self.L.otz_extract_run(self.h, plan, d_archive, archive_len, d_out, out_len), "otz_extract_run")

    def results(self, plan, n: int):
        crc = np.zeros(max(n, 1), dtype=np.uint32)
        st = np.zeros(max(n, 1), dtype=np.int32)
        self.lib.check(self.L.otz_extract_results(self.h, plan, crc.ctypes.data_as(C.c_void_p),
                                                  st.ctypes.data_as(C.c_void_p)), "otz_extract_results")
        return crc[:n], st[:n]

    def extract_host(self, img, table: np.ndarray, opts: OtzOpts | None = None):
        """H2D image -> batch extract -> D2H arena. -> (out uint8[], crc uint32[n], status int32[n])"""
        opts = opts or default_opts()
        n = len(table)
        t = np.ascontiguousarray(table)
        out_len = int((t["out_ofs"].astype(np.int64) + t["uncomp_size"]).max()) if n else 0
        out = np.zeros(max(out_len, 1), dtype=np.uint8)
        crc = np.zeros(max(n, 1), dtype=np.uint32)
        st = np.zeros(max(n, 1), dtype=np.int32)
        buf = np.frombuffer(img, dtype=np.uint8) if not isinstance(img, np.ndarray) else img
        self.lib.check(self.L.otz_extract_host(self.h, buf.ctypes.data_as(C.c_void_p), buf.nbytes,
                                               t.ctypes.data_as(C.c_void_p), n, C.byref(opts),
                                               out.ctypes.data_as(C.c_void_p), out_len,
                                               crc.ctypes.data_as(C.c_void_p), st.ctypes.data_as(C.c_void_p)),
                       "otz_extract_host")
        return out[:out_len], crc[:n], st[:n]

    # -- write path
    def deflate_host(self, sources: list, methods: list | None = None):
        """Batched otezip_compress_data + CRC through the C-ABI host-buffer call.
        -> list of (method_out, payload bytes, crc32)"""
        n = len(sources)
        methods = methods or [8] * n
        lens = np.array([len(s) for s in sources], dtype=np.uint32)
        ofs = np.zeros(n, dtype=np.uint64)
        pos = 0
        for i in range(n):
            ofs[i] = pos
            pos += (int(lens[i]) + 15) & ~15
        buf = np.zeros(max(pos, 1), dtype=np.uint8)
        for i, s in enumerate(sources):
            buf[int(ofs[i]):int(ofs[i]) + len(s)] = np.frombuffer(s, dtype=np.uint8)
        meth = np.array(methods, dtype=np.uint16)
        out = np.zeros(max(int(lens.astype(np.int64).sum()), 1), dtype=np.uint8)
        o_ofs = np.zeros(max(n, 1), dtype=np.uint64)
        o_sz = np.zeros(max(n, 1), dtype=np.uint32)
        crc = np.zeros(max(n, 1), dtype=np.uint32)
        m_out = np.zeros(max(n, 1), dtype=np.uint16)
        tot = C.c_uint64()
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self.lib.check(self.L.otz_deflate_host(self.h, vp(buf), pos, vp(ofs), vp(lens), vp(meth), n, vp(out), out.nbytes,
                                               vp(o_ofs), vp(o_sz), vp(crc), vp(m_out), C.byref(tot)), "otz_deflate_host")
        return [(int(m_out[i]), bytes(out[int(o_ofs[i]):int(o_ofs[i]) + int(o_sz[i])]), int(crc[i])) for i in range(n)]

    # -- write path, device-resident (what bench.py times)
    def deflate_plan(self, in_ofs: np.ndarray, in_len: np.ndarray, methods: np.ndarray):
        j = C.c_void_p()
        vp = lambda a: np.ascontiguousarray(a).ctypes.data_as(C.c_void_p)
        self._dfl_keep = (np.ascontiguousarray(in_ofs, dtype=np.uint64), np.ascontiguousarray(in_len, dtype=np.uint32),
                          np.ascontiguousarray(methods, dtype=np.uint16))
        a, b, c = self._dfl_keep
        self.lib.check(self.L.otz_deflate_plan(self.h, a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p),
                                               c.ctypes.data_as(C.c_void_p), len(a), C.byref(j)), "otz_deflate_plan")
        return j

    def deflate_run(self, job, d_in, in_bytes: int):
        self.lib.check(self.L.otz_deflate_run(self.h, job, d_in, in_bytes), "otz_deflate_run")

    def deflate_results(self, job, n: int):
        ofs = np.zeros(max(n, 1), dtype=np.uint64)
        sz = np.zeros(max(n, 1), dtype=np.uint32)
        crc = np.zeros(max(n, 1), dtype=np.uint32)
        m = np.zeros(max(n, 1), dtype=np.uint16)
        tot = C.c_uint64()
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self.lib.check(self.L.otz_deflate_results(self.h, job, vp(ofs), vp(sz), vp(crc), vp(m), C.byref(tot)), "otz_deflate_results")
        return ofs[:n], sz[:n], crc[:n], m[:n], int(tot.value)

    def deflate_fetch(self, job, nbytes: int) -> np.ndarray:
        out = np.zeros(max(nbytes, 1), dtype=np.uint8)
        self.lib.check(self.L.otz_deflate_fetch(self.h, job, out.ctypes.data_as(C.c_void_p), nbytes), "otz_deflate_fetch")
        return out[:nbytes]

    def deflate_destroy(self, job):
        self.L.otz_deflate_destroy(self.h, job)

    def deflate_chunks(self, job, n: int):
        """-> (first_chunk[n], n_chunks[n], csize[total], chunk_bytes)"""
        first = np.zeros(max(n, 1), dtype=np.uint32)
        cnt = np.zeros(max(n, 1), dtype=np.uint32)
        cb = C.c_uint32()
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        tot = self.L.otz_deflate_chunks(self.h, job, vp(first), vp(cnt), None, 0, C.byref(cb))
        if tot < 0:
            self.lib.check(tot, "otz_deflate_chunks")
        cs = np.zeros(max(tot, 1), dtype=np.uint32)
        if tot:
            r = self.L.otz_deflate_chunks(self.h, job, None, None, vp(cs), tot, None)
            if r < 0:
                self.lib.check(r, "otz_deflate_chunks")
        return first[:n], cnt[:n], cs[:tot], int(cb.value)

    # -- WinZip AES (device-resident buffers; what tools/aes_bench.py times)
    @staticmethod
    def _passwords(passwords):
        arr = (C.c_char_p * max(len(passwords), 1))(*[p if isinstance(p, bytes) else p.encode() for p in passwords])
        return arr, len(passwords)

    def aes_open(self, d_src, src_len: int, rows: np.ndarray, passwords, d_plain, plain_len: int):
        """Asynchronous: KDF + CTR into the plaintext image, MAC on the side stream.  rows: AES_ENTRY_DTYPE."""
        r = np.ascontiguousarray(rows, dtype=AES_ENTRY_DTYPE)
        pw, n_pw = self._passwords(passwords)
        self._aes_keep = (r, pw)
        self.lib.check(self.L.otz_aes_open(self.h, d_src, src_len, r.ctypes.data_as(C.c_void_p), len(r), pw, n_pw, d_plain, plain_len),
                       "otz_aes_open")

    def aes_status(self, n: int) -> np.ndarray:
        st = np.zeros(max(n, 1), dtype=np.int32)
        self.lib.check(self.L.otz_aes_status(self.h, st.ctypes.data_as(C.c_void_p)), "otz_aes_status")
        return st[:n]

    def aes_times(self):
        """-> (ms_kdf, ms_ctr, ms_mac) of the last aes_open"""
        f = [C.c_float() for _ in range(3)]
        self.lib.check(self.L.otz_aes_times(self.h, *[C.byref(x) for x in f]), "otz_aes_times")
        return tuple(x.value for x in f)

    def aes_seal(self, d_in, in_len: int, rows: np.ndarray, salts: bytes, passwords, d_out, out_len: int):
        r = np.ascontiguousarray(rows, dtype=AES_ENTRY_DTYPE)
        pw, n_pw = self._passwords(passwords)
        sb = np.frombuffer(salts, dtype=np.uint8)
        assert sb.size >= 16 * len(r)
        self.lib.check(self.L.otz_aes_seal(self.h, d_in, in_len, r.ctypes.data_as(C.c_void_p), len(r), sb.ctypes.data_as(C.c_void_p),
                                           pw, n_pw, d_out, out_len), "otz_aes_seal")

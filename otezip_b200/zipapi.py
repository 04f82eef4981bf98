"""ctypes view of the libzip-subset API exported by libotezip_b200.so (include/otezip/zip.h) — the same
calls, names and argument meaning as the reference's src/include/otezip/zip.h:192-215, so the parity
tests read like the reference's own tests.  No logic lives here."""
from __future__ import annotations

import ctypes as C

from .native import Lib

ZIP_RDONLY, ZIP_CREATE, ZIP_EXCL, ZIP_TRUNCATE = 0, 1, 2, 8
ZIP_CM_STORE, ZIP_CM_DEFLATE, ZIP_CM_DEFLATE64, ZIP_CM_XZ = 0, 8, 9, 95
ZIP_EM_NONE, ZIP_EM_TRAD_PKWARE, ZIP_EM_AES_128, ZIP_EM_AES_192, ZIP_EM_AES_256 = 0, 1, 0x0101, 0x0102, 0x0103


class ZipFileT(C.Structure):  # struct zip_file
    _fields_ = [("data", C.POINTER(C.c_uint8)), ("size", C.c_uint32), ("pos", C.c_uint64)]


class ZipEntry(C.Structure):  # struct otezip_entry
    _fields_ = [("name", C.c_char_p), ("local_hdr_ofs", C.c_uint32), ("comp_size", C.c_uint32),
                ("uncomp_size", C.c_uint32), ("method", C.c_uint16), ("crc32", C.c_uint32),
                ("file_time", C.c_uint16), ("file_date", C.c_uint16), ("external_attr", C.c_uint32)]


class ZipT(C.Structure):  # struct zip
    _fields_ = [("fp", C.c_void_p), ("entries", C.POINTER(ZipEntry)), ("n_entries", C.c_uint64), ("mode", C.c_int),
                ("next_index", C.c_uint64), ("default_method", C.c_uint16)]


class ZipStat(C.Structure):  # struct zip_stat
    _fields_ = [("valid", C.c_uint64), ("name", C.c_char_p), ("index", C.c_uint64), ("size", C.c_uint64),
                ("comp_size", C.c_uint64), ("mtime", C.c_long), ("crc", C.c_uint32), ("comp_method", C.c_uint16)]


class ZipApi:
    def __init__(self, cdll=None):
        L = self.L = cdll or Lib.get().L
        P = C.POINTER
        L.zip_open.restype = P(ZipT)
        L.zip_open.argtypes = [C.c_char_p, C.c_int, P(C.c_int)]
        L.zip_close.argtypes = [P(ZipT)]
        L.zip_get_num_files.restype = C.c_uint64
        L.zip_get_num_files.argtypes = [P(ZipT)]
        L.zip_get_name.restype = C.c_char_p
        L.zip_get_name.argtypes = [P(ZipT), C.c_uint64, C.c_int]
        L.zip_name_locate.restype = C.c_int64
        L.zip_name_locate.argtypes = [P(ZipT), C.c_char_p, C.c_int]
        L.zip_fopen_index.restype = P(ZipFileT)
        L.zip_fopen_index.argtypes = [P(ZipT), C.c_uint64, C.c_int]
        L.zip_fclose.argtypes = [P(ZipFileT)]
        L.zip_fread.restype = C.c_int64
        L.zip_fread.argtypes = [P(ZipFileT), C.c_void_p, C.c_uint64]
        L.zip_stat_index.argtypes = [P(ZipT), C.c_uint64, C.c_int, P(ZipStat)]
        L.zip_stat_init.argtypes = [P(ZipStat)]
        L.zip_stat_init.restype = None
        L.zip_source_buffer.restype = C.c_void_p
        L.zip_source_buffer.argtypes = [P(ZipT), C.c_void_p, C.c_uint64, C.c_int]
        L.zip_source_free.argtypes = [C.c_void_p]
        L.zip_source_free.restype = None
        L.zip_file_add.restype = C.c_int64
        L.zip_file_add.argtypes = [P(ZipT), C.c_char_p, C.c_void_p, C.c_int]
        L.zip_set_file_compression.argtypes = [P(ZipT), C.c_uint64, C.c_int32, C.c_uint32]
        L.zip_file_replace.argtypes = [P(ZipT), C.c_uint64, C.c_void_p, C.c_int]
        L.otezip_method_from_string.argtypes = [C.c_char_p]
        L.zip_set_default_password.argtypes = [P(ZipT), C.c_char_p]
        L.zip_fopen_index_encrypted.restype = P(ZipFileT)
        L.zip_fopen_index_encrypted.argtypes = [P(ZipT), C.c_uint64, C.c_int, C.c_char_p]
        L.zip_file_set_encryption.argtypes = [P(ZipT), C.c_uint64, C.c_uint16, C.c_char_p]
        L.zip_encryption_method_supported.argtypes = [C.c_uint16, C.c_int]
        L.zip_compression_method_supported.argtypes = [C.c_int32, C.c_int]
        L.otezip_b200_entry_status.argtypes = [P(ZipT), C.c_uint64]
        self.verify_crc = C.c_int.in_dll(L, "otezip_verify_crc")
        self.ignore_zipbomb = C.c_int.in_dll(L, "otezip_ignore_zipbomb")
        try:
            self.ref_compat = C.c_int.in_dll(L, "otezip_ref_compat")
        except ValueError:  # the compiled reference has no such switch
            self.ref_compat = None

    # -- helpers written as a libzip consumer would write them
    def read_all(self, path: str, verify_crc: int = 1):
        """zip_open -> zip_fopen_index(i) -> zip_fread -> zip_fclose.  -> (err, names, [bytes|None])"""
        self.verify_crc.value = verify_crc
        err = C.c_int(-99)
        za = self.L.zip_open(path.encode(), ZIP_RDONLY, C.byref(err))
        if not za:
            return err.value, None, None
        n = self.L.zip_get_num_files(za)
        names, datas = [], []
        for i in range(n):
            names.append(self.L.zip_get_name(za, i, 0))
            zf = self.L.zip_fopen_index(za, i, 0)
            if not zf:
                datas.append(None)
                continue
            size = zf.contents.size
            buf = C.create_string_buffer(max(size, 1))
            got = self.L.zip_fread(zf, buf, size)
            assert got == size and self.L.zip_fread(zf, buf, 1) == 0
            datas.append(buf.raw[:size])
            self.L.zip_fclose(zf)
        assert self.L.zip_close(za) == 0
        return err.value, names, datas

    def write_archive(self, path: str, files, method: int | None = ZIP_CM_DEFLATE, use_default_method: bool = False):
        """files: list of (name, bytes[, method[, level]]).  Per-file method (and libzip compression level) via zip_set_file_compression after
        zip_file_add (README.md:33-55 idiom) or via za->default_method (what main.c:188-191 does)."""
        libc = C.CDLL(None)
        libc.malloc.restype = C.c_void_p
        libc.malloc.argtypes = [C.c_size_t]
        err = C.c_int(-99)
        za = self.L.zip_open(path.encode(), ZIP_CREATE | ZIP_TRUNCATE, C.byref(err))
        assert za, err.value
        if use_default_method and method is not None:
            za.contents.default_method = method
        for f in files:
            name, data = f[0], f[1]
            m = f[2] if len(f) > 2 else method
            p = libc.malloc(max(len(data), 1))
            C.memmove(p, data, len(data))
            src = self.L.zip_source_buffer(za, p, len(data), 1)          # freep=1: the library owns p
            idx = self.L.zip_file_add(za, name.encode(), src, 0)
            assert idx >= 0
            if not use_default_method and m is not None:
                assert self.L.zip_set_file_compression(za, idx, m, f[3] if len(f) > 3 else 0) == 0
        return self.L.zip_close(za)

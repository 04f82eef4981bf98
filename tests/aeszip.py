"""WinZip AES (AE-1 / AE-2, method 99) writer and reader used by the tests as an independent reference.

It imports nothing of the library: AES is written here in numpy (vectorised over counter blocks, S-box derived from the
GF(2^8) inverse rather than copied), PBKDF2 and HMAC come from hashlib / hmac, and the ZIP records are packed with struct.
No third-party AES archiver is available to compare against, so interoperability rests on the published format, which
the known-answer vectors in tests/test_aes_cpu.py pin (FIPS-197, NIST SP 800-38A, RFC 6070)."""
from __future__ import annotations

import hashlib
import hmac
import os
import struct
import zlib
from dataclasses import dataclass

import numpy as np


def _gf_mul(a: int, b: int) -> int:
    p = 0
    while b:
        if b & 1:
            p ^= a
        a = ((a << 1) ^ 0x11B) if a & 0x80 else a << 1
        b >>= 1
    return p


def _sbox() -> np.ndarray:
    s = np.zeros(256, dtype=np.uint8)
    for x in range(256):
        inv = 0
        if x:
            inv = 1
            for _ in range(254):          # x^254 = x^-1
                inv = _gf_mul(inv, x)
        b = inv
        r = b
        for k in range(1, 5):
            r ^= ((b << k) | (b >> (8 - k))) & 0xFF
        s[x] = r ^ 0x63
    return s


SBOX = _sbox()
XT2 = np.array([_gf_mul(x, 2) for x in range(256)], dtype=np.uint8)
XT3 = np.array([_gf_mul(x, 3) for x in range(256)], dtype=np.uint8)
# ShiftRows on the column-major state (byte r + 4c): new[r + 4c] = old[r + 4((c + r) % 4)]
SHIFT = np.array([r + 4 * ((c + r) % 4) for c in range(4) for r in range(4)])


def expand_key(key: bytes) -> np.ndarray:
    """FIPS-197 key expansion -> round keys as uint8[(Nr + 1), 16]."""
    nk = len(key) // 4
    assert nk in (4, 6, 8)
    nr = nk + 6
    w = [list(key[4 * i:4 * i + 4]) for i in range(nk)]
    rcon = 1
    for i in range(nk, 4 * (nr + 1)):
        t = list(w[i - 1])
        if i % nk == 0:
            t = t[1:] + t[:1]
            t = [int(SBOX[b]) for b in t]
            t[0] ^= rcon
            rcon = _gf_mul(rcon, 2)
        elif nk > 6 and i % nk == 4:
            t = [int(SBOX[b]) for b in t]
        w.append([a ^ b for a, b in zip(w[i - nk], t)])
    return np.array(w, dtype=np.uint8).reshape(nr + 1, 16)


def aes_encrypt_blocks(key: bytes, blocks: np.ndarray) -> np.ndarray:
    """AES encryption of uint8[N, 16] blocks."""
    rk = expand_key(key)
    s = blocks.astype(np.uint8) ^ rk[0]
    for r in range(1, len(rk)):
        s = SBOX[s][:, SHIFT]
        if r != len(rk) - 1:
            c = s.reshape(-1, 4, 4)   # [block, column, row]
            a0, a1, a2, a3 = c[:, :, 0], c[:, :, 1], c[:, :, 2], c[:, :, 3]
            s = np.stack([XT2[a0] ^ XT3[a1] ^ a2 ^ a3, a0 ^ XT2[a1] ^ XT3[a2] ^ a3,
                          a0 ^ a1 ^ XT2[a2] ^ XT3[a3], XT3[a0] ^ a1 ^ a2 ^ XT2[a3]], axis=2).reshape(-1, 16)
        s = s ^ rk[r]
    return s


def ctr_winzip(key: bytes, data: bytes) -> bytes:
    """AES-CTR as WinZip AES uses it: little-endian 128-bit counter starting at 1."""
    n = (len(data) + 15) // 16
    if n == 0:
        return b""
    blocks = np.zeros((n, 16), dtype=np.uint8)
    blocks[:, :8] = np.arange(1, n + 1, dtype="<u8").view(np.uint8).reshape(n, 8)
    ks = aes_encrypt_blocks(key, blocks).reshape(-1)[:len(data)]
    return (np.frombuffer(data, dtype=np.uint8) ^ ks).tobytes()


KEYLEN = {1: 16, 2: 24, 3: 32}


def derive(password: bytes, salt: bytes, strength: int):
    kl = KEYLEN[strength]
    dk = hashlib.pbkdf2_hmac("sha1", password, salt, 1000, 2 * kl + 2)
    return dk[:kl], dk[kl:2 * kl], dk[2 * kl:]


def seal(payload: bytes, password: bytes, strength: int, salt: bytes | None = None) -> bytes:
    """salt | verification value | ciphertext | authentication code"""
    salt = salt if salt is not None else os.urandom(4 + 4 * strength)
    assert len(salt) == 4 + 4 * strength
    key, mkey, pwv = derive(password, salt, strength)
    ct = ctr_winzip(key, payload)
    return salt + pwv + ct + hmac.new(mkey, ct, hashlib.sha1).digest()[:10]


class AuthError(ValueError):
    pass


def open_payload(blob: bytes, password: bytes, strength: int) -> bytes:
    sl = 4 + 4 * strength
    salt, pwv, ct, mac = blob[:sl], blob[sl:sl + 2], blob[sl + 2:-10], blob[-10:]
    key, mkey, want = derive(password, salt, strength)
    if pwv != want:
        raise AuthError("wrong password")
    if not hmac.compare_digest(hmac.new(mkey, ct, hashlib.sha1).digest()[:10], mac):
        raise AuthError("authentication code mismatch")
    return ctr_winzip(key, ct)


@dataclass
class Entry:
    name: str
    method: int              # actual compression method (0 / 8 / 93)
    payload: bytes           # compressed bytes
    uncomp_size: int
    crc32: int               # CRC-32 of the plaintext
    strength: int = 0        # 0 = stored unencrypted
    vendor: int = 2          # 1 = AE-1 (CRC stored), 2 = AE-2 (CRC field 0)
    password: bytes = b""
    salt: bytes | None = None


def build_zip(entries: list[Entry]) -> bytes:
    """A ZIP image; encrypted entries get method 99, flag bit 0 and the 0x9901 field in both headers."""
    out, cd = bytearray(), bytearray()
    for e in entries:
        name = e.name.encode()
        if e.strength:
            data = seal(e.payload, e.password, e.strength, e.salt)
            x = struct.pack("<HHH2sBH", 0x9901, 7, e.vendor, b"AE", e.strength, e.method)
            method, flags, crc = 99, 1, (e.crc32 if e.vendor == 1 else 0)
        else:
            data, x, method, flags, crc = e.payload, b"", e.method, 0, e.crc32
        ofs = len(out)
        out += struct.pack("<IHHHHHIIIHH", 0x04034B50, 20, flags, method, 0, 0x21, crc, len(data), e.uncomp_size, len(name), len(x))
        out += name + x + data
        cd += struct.pack("<IHHHHHHIIIHHHHHII", 0x02014B50, 0x031E, 20, flags, method, 0, 0x21, crc, len(data), e.uncomp_size,
                          len(name), len(x), 0, 0, 0, 0o100644 << 16, ofs)
        cd += name + x
    cd_ofs = len(out)
    out += cd
    n = len(entries)
    out += struct.pack("<IHHHHIIH", 0x06054B50, 0, 0, n, n, len(cd), cd_ofs, 0)
    return bytes(out)


def read_zip(img: bytes, password: bytes | None = None) -> list[dict]:
    """Directory walk (ZIP32 and ZIP64 extras) plus, with a password, the decrypted compressed bytes of every entry."""
    p = img.rfind(b"PK\x05\x06")
    n, cd_size, cd_ofs = struct.unpack_from("<HII", img, p + 10)
    if n == 0xFFFF or cd_ofs == 0xFFFFFFFF:
        rpos = struct.unpack_from("<Q", img, p - 12)[0]
        n, cd_size, cd_ofs = struct.unpack_from("<QQQ", img, rpos + 32)
    res, off = [], cd_ofs
    for _ in range(n):
        (sig, _, _, flags, method, _, _, crc, comp, uncomp, fl, xl, cl, _, _, _, lfh) = struct.unpack_from("<IHHHHHHIIIHHHHHII", img, off)
        assert sig == 0x02014B50
        name = img[off + 46:off + 46 + fl].decode()
        x = img[off + 46 + fl:off + 46 + fl + xl]
        d = dict(name=name, flags=flags, method=method, crc32=crc, comp_size=comp, uncomp_size=uncomp, lfh=lfh, aes=None)
        o = 0
        while o + 4 <= len(x):
            hid, sz = struct.unpack_from("<HH", x, o)
            if hid == 1 and lfh == 0xFFFFFFFF:
                d["lfh"] = lfh = struct.unpack_from("<Q", x, o + 4)[0]
            if hid == 0x9901:
                ver, ae, st, am = struct.unpack_from("<H2sBH", x, o + 4)
                d["aes"] = dict(vendor=ver, strength=st, method=am)
            o += 4 + sz
        nl, lxl = struct.unpack_from("<HH", img, lfh + 26)
        data = img[lfh + 30 + nl + lxl:lfh + 30 + nl + lxl + comp]
        d["local_flags"], d["local_method"] = struct.unpack_from("<HH", img, lfh + 6)
        d["raw"] = data
        if d["aes"] and password is not None:
            d["payload"] = open_payload(data, password, d["aes"]["strength"])
        res.append(d)
        off += 46 + fl + xl + cl
    return res


def inflate(method: int, payload: bytes) -> bytes:
    if method == 0:
        return payload
    if method == 8:
        return zlib.decompress(payload, -15)
    raise ValueError(method)

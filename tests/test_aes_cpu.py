"""WinZip AES without a device: the tests' reference (tests/aeszip.py) against published known answers, and what the library
answers about encrypted archives before anything is decoded."""
import ctypes as C
import hashlib
import zlib

import numpy as np
import pytest

from tests import aeszip

PT = bytes.fromhex("00112233445566778899aabbccddeeff")


@pytest.mark.parametrize("key,ct", [
    ("000102030405060708090a0b0c0d0e0f", "69c4e0d86a7b0430d8cdb78070b4c55a"),                                   # FIPS-197 C.1
    ("000102030405060708090a0b0c0d0e0f1011121314151617", "dda97ca4864cdfe06eaf70a0ec0d7191"),                   # C.2
    ("000102030405060708090a0b0c0d0e0f101112131415161718191a1b1c1d1e1f", "8ea2b7ca516745bfeafc49904b496089"),   # C.3
])
def test_aes_fips197_appendix_c(key, ct):
    out = aeszip.aes_encrypt_blocks(bytes.fromhex(key), np.frombuffer(PT, dtype=np.uint8).reshape(1, 16))
    assert out.tobytes().hex() == ct


SP800_PT = bytes.fromhex("6bc1bee22e409f96e93d7e117393172aae2d8a571e03ac9c9eb76fac45af8e51"
                         "30c81c46a35ce411e5fbc1191a0a52eff69f2445df4f9b17ad2b417be66c3710")


@pytest.mark.parametrize("key,ct", [
    ("2b7e151628aed2a6abf7158809cf4f3c",                                                                          # F.5.1
     "874d6191b620e3261bef6864990db6ce9806f66b7970fdff8617187bb9fffdff5ae4df3edbd5d35e5b4f09020db03eab1e031dda2fbe03d1792170a0f3009cee"),
    ("8e73b0f7da0e6452c810f32b809079e562f8ead2522c6b7b",                                                          # F.5.3
     "1abc932417521ca24f2b0459fe7e6e0b090339ec0aa6faefd5ccc2c6f4ce8e941e36b26bd1ebc670d1bd1d665620abf74f78a7f6d29809585a97daec58c6b050"),
    ("603deb1015ca71be2b73aef0857d77811f352c073b6108d72d9810a30914dff4",                                          # F.5.5
     "601ec313775789a5b7a7f504bbf3d228f443e3ca4d62b59aca84e990cacaf5c52b0930daa23de94ce87017ba2d84988ddfc9c58db67aada613c2dd08457941a6"),
])
def test_aes_ctr_sp800_38a_f5(key, ct):
    # SP 800-38A counts big-endian from f0f1..ff; WinZip counts little-endian from 1 — the block cipher is the same
    ctr = int.from_bytes(bytes.fromhex("f0f1f2f3f4f5f6f7f8f9fafbfcfdfeff"), "big")
    blocks = np.frombuffer(b"".join(((ctr + i) % (1 << 128)).to_bytes(16, "big") for i in range(4)), dtype=np.uint8).reshape(4, 16)
    ks = aeszip.aes_encrypt_blocks(bytes.fromhex(key), blocks).reshape(-1)
    assert (np.frombuffer(SP800_PT, dtype=np.uint8) ^ ks).tobytes().hex() == ct


@pytest.mark.parametrize("pw,salt,c,n,dk", [
    (b"password", b"salt", 1, 20, "0c60c80f961f0e71f3a9b524af6012062fe037a6"),
    (b"password", b"salt", 2, 20, "ea6c014dc72d6f8ccd1ed92ace1d41f0d8de8957"),
    (b"password", b"salt", 4096, 20, "4b007901b765489abead49d926f721d065a429c1"),
    (b"passwordPASSWORDpassword", b"saltSALTsaltSALTsaltSALTsaltSALTsalt", 4096, 25, "3d2eec4fe41c849b80c8d83662c0e44a8b291a964cf2f07038"),
])
def test_pbkdf2_rfc6070(pw, salt, c, n, dk):
    assert hashlib.pbkdf2_hmac("sha1", pw, salt, c, n).hex() == dk


def test_winzip_counter_is_little_endian_from_one():
    key = bytes(range(16))
    ks = aeszip.ctr_winzip(key, bytes(48))
    blocks = np.zeros((3, 16), dtype=np.uint8)
    blocks[:, 0] = [1, 2, 3]
    assert ks == aeszip.aes_encrypt_blocks(key, blocks).tobytes()


@pytest.mark.parametrize("strength", [1, 2, 3])
def test_helper_round_trip_and_tamper(strength):
    data = zlib.compress(b"hello AES " * 100)
    blob = aeszip.seal(data, b"pw", strength)
    assert len(blob) == len(data) + 4 + 4 * strength + 12
    assert aeszip.open_payload(blob, b"pw", strength) == data
    with pytest.raises(aeszip.AuthError):
        aeszip.open_payload(blob, b"wrong", strength)
    bad = bytearray(blob)
    bad[4 + 4 * strength + 2] ^= 1
    with pytest.raises(aeszip.AuthError):
        aeszip.open_payload(bytes(bad), b"pw", strength)


def test_zip_open_lists_encrypted_entries_without_device(tmp_path):
    from otezip_b200.zipapi import ZipApi, ZipStat
    api = ZipApi()
    raw = [b"alpha " * 300, b"", b"\x00\x01" * 5000]
    ents = [aeszip.Entry("a.txt", 8, zlib.compress(raw[0])[2:-4], len(raw[0]), zlib.crc32(raw[0]), 3, 2, b"secret"),
            aeszip.Entry("b.empty", 0, b"", 0, 0, 1, 1, b"secret"),
            aeszip.Entry("c.bin", 0, raw[2], len(raw[2]), zlib.crc32(raw[2]), 2, 1, b"secret"),
            aeszip.Entry("d.plain", 0, raw[0], len(raw[0]), zlib.crc32(raw[0]))]
    img = aeszip.build_zip(ents)
    p = tmp_path / "enc.zip"
    p.write_bytes(img)
    err = C.c_int(-1)
    za = api.L.zip_open(str(p).encode(), 0, C.byref(err))
    assert za and err.value == 0
    assert api.L.zip_get_num_files(za) == 4
    st = ZipStat()
    for i, e in enumerate(ents):
        assert api.L.zip_stat_index(za, i, 0, C.byref(st)) == 0
        assert st.name.decode() == e.name and st.size == e.uncomp_size
        assert st.comp_method == (99 if e.strength else e.method)
        assert st.comp_size == len(e.payload) + (4 + 4 * e.strength + 12 if e.strength else 0)
        assert st.crc == (0 if e.strength and e.vendor == 2 else e.crc32)
    assert api.L.zip_set_default_password(za, b"x") == 0 and api.L.zip_set_default_password(za, None) == 0
    assert api.L.zip_close(za) == 0


def test_encryption_method_supported():
    from otezip_b200.zipapi import ZipApi, ZIP_EM_NONE, ZIP_EM_TRAD_PKWARE, ZIP_EM_AES_128, ZIP_EM_AES_192, ZIP_EM_AES_256
    L = ZipApi().L
    for enc in (0, 1):
        assert L.zip_encryption_method_supported(ZIP_EM_NONE, enc) == 1
        for m in (ZIP_EM_AES_128, ZIP_EM_AES_192, ZIP_EM_AES_256):
            assert L.zip_encryption_method_supported(m, enc) == 1
        for m in (ZIP_EM_TRAD_PKWARE, 2, 0x0104, 0x6601):
            assert L.zip_encryption_method_supported(m, enc) == 0


def test_set_encryption_refuses_unsupported_and_on_disk_entries(tmp_path):
    from otezip_b200.zipapi import ZipApi, ZIP_CREATE, ZIP_TRUNCATE, ZIP_EM_NONE, ZIP_EM_AES_256, ZIP_EM_TRAD_PKWARE
    L = ZipApi().L
    err = C.c_int(-1)
    # an entry added in this session, in write mode: only the unsupported methods are refused
    za = L.zip_open(str(tmp_path / "new.zip").encode(), ZIP_CREATE | ZIP_TRUNCATE, C.byref(err))
    assert za and za.contents.mode == 1
    data = C.create_string_buffer(b"abc", 3)
    i = L.zip_file_add(za, b"new", L.zip_source_buffer(za, data, 3, 0), 0)
    assert i == 0
    for m in (ZIP_EM_TRAD_PKWARE, 2, 0x0104):
        assert L.zip_file_set_encryption(za, i, m, b"pw") == -1, m
    assert L.zip_file_set_encryption(za, i, ZIP_EM_AES_256, b"pw") == 0
    assert L.zip_file_set_encryption(za, i, ZIP_EM_NONE, None) == 0
    assert L.zip_file_set_encryption(za, 5, ZIP_EM_AES_256, b"pw") == -1          # no such entry
    za.contents.mode = 0   # close without writing (writing needs a device)
    L.zip_close(za)
    # an entry already on disk (append mode): refused whatever the method
    p = tmp_path / "x.zip"
    p.write_bytes(aeszip.build_zip([aeszip.Entry("old", 0, b"abc", 3, zlib.crc32(b"abc"))]))
    za = L.zip_open(str(p).encode(), ZIP_CREATE, C.byref(err))
    assert za and za.contents.mode == 1
    assert L.zip_file_set_encryption(za, 0, ZIP_EM_AES_256, b"pw") == -1
    za.contents.mode = 0
    L.zip_close(za)

// k_aes.cuh — WinZip AES (AE-1 / AE-2, method 99) on the device: key derivation, AES-CTR and HMAC-SHA1.
//
// An encrypted entry's payload is  salt (8/12/16) | password verification value (2) | ciphertext | authentication code (10).
//   k_aes_kdf  PBKDF2-HMAC-SHA1(password, salt, 1000, 2*keylen + 2): one lane per (entry, 20-byte output block T_i), four
//              lanes reserved per entry (AES-128 uses 2, -192 3, -256 4).  The lane absorbs the password's ipad / opad blocks
//              once; each iteration is then two SHA-1 compressions with the state in registers.  Lane 0 of the entry then
//              checks (open) or writes (seal) the verification value and expands the AES round keys, lane 1 absorbs the
//              HMAC key into its inner / outer SHA-1 states.
//   k_aes_ctr  AES-CTR, little-endian 128-bit counter starting at 1 (only the low 32 bits change: entries are < 2 GiB).
//              One CTA per (entry, 64 KiB chunk) of a work list; T-tables and round keys in shared memory; one 16-byte
//              block per thread and step, loaded and stored as one 16-byte vector when both sides are aligned.  CTR is
//              symmetric, so the same kernel decrypts (open: into a plaintext image whose entries start with a synthetic
//              30-byte local header) and encrypts (seal).
//   k_aes_mac  HMAC-SHA1 over the ciphertext, one lane per entry, longest entry first.  The chain is serial by construction.
//              Open compares the first 10 bytes in constant time; seal writes them.
#pragma once
#include "otz_common.cuh"

#define OTZ_AES_CHUNK 65536u        // ciphertext bytes per CTR work item
#define OTZ_AES_CTR_THREADS 256
#define OTZ_AES_KDF_THREADS 128     // 32 entries per CTA
#define OTZ_AES_ITER 1000
#define OTZ_AES_NOPW 0xFFFFu

// One row per entry, built by the host side of otz_aes_open / otz_aes_seal.  Offsets are in the buffers the kernels take.
struct OtzAesJob {
	uint64_t salt;       // salt (in the source for open, in the salt array for seal)
	uint64_t pwv;        // 2-byte verification value (source for open, output for seal)
	uint64_t src;        // first input byte of CTR (ciphertext for open, plaintext for seal)
	uint64_t dst;        // first output byte of CTR
	uint64_t mac;        // 10-byte authentication code (source for open, output for seal)
	uint64_t hdr;        // open: synthetic local header in the plaintext image; seal: salt destination in the output
	uint32_t len;        // ciphertext bytes
	uint16_t strength;   // 1 / 2 / 3 = AES-128 / 192 / 256
	uint16_t pw;         // password index, OTZ_AES_NOPW = none
};

struct OtzAesWork {
	uint32_t job, chunk;
};

// Derived per-entry key material (device scratch, cleared at the end of every run).
struct OtzAesKeys {
	uint32_t rk[60];     // expanded encryption key, FIPS-197 word order
	uint32_t hi[5], ho[5];   // HMAC-SHA1 states after the key's ipad / opad block
	uint32_t nr;         // rounds
	uint32_t pad_;
};

__device__ const uint8_t g_aes_sbox[256] = {
	0x63, 0x7c, 0x77, 0x7b, 0xf2, 0x6b, 0x6f, 0xc5, 0x30, 0x01, 0x67, 0x2b, 0xfe, 0xd7, 0xab, 0x76, 0xca, 0x82, 0xc9, 0x7d, 0xfa, 0x59, 0x47,
	0xf0, 0xad, 0xd4, 0xa2, 0xaf, 0x9c, 0xa4, 0x72, 0xc0, 0xb7, 0xfd, 0x93, 0x26, 0x36, 0x3f, 0xf7, 0xcc, 0x34, 0xa5, 0xe5, 0xf1, 0x71, 0xd8,
	0x31, 0x15, 0x04, 0xc7, 0x23, 0xc3, 0x18, 0x96, 0x05, 0x9a, 0x07, 0x12, 0x80, 0xe2, 0xeb, 0x27, 0xb2, 0x75, 0x09, 0x83, 0x2c, 0x1a, 0x1b,
	0x6e, 0x5a, 0xa0, 0x52, 0x3b, 0xd6, 0xb3, 0x29, 0xe3, 0x2f, 0x84, 0x53, 0xd1, 0x00, 0xed, 0x20, 0xfc, 0xb1, 0x5b, 0x6a, 0xcb, 0xbe, 0x39,
	0x4a, 0x4c, 0x58, 0xcf, 0xd0, 0xef, 0xaa, 0xfb, 0x43, 0x4d, 0x33, 0x85, 0x45, 0xf9, 0x02, 0x7f, 0x50, 0x3c, 0x9f, 0xa8, 0x51, 0xa3, 0x40,
	0x8f, 0x92, 0x9d, 0x38, 0xf5, 0xbc, 0xb6, 0xda, 0x21, 0x10, 0xff, 0xf3, 0xd2, 0xcd, 0x0c, 0x13, 0xec, 0x5f, 0x97, 0x44, 0x17, 0xc4, 0xa7,
	0x7e, 0x3d, 0x64, 0x5d, 0x19, 0x73, 0x60, 0x81, 0x4f, 0xdc, 0x22, 0x2a, 0x90, 0x88, 0x46, 0xee, 0xb8, 0x14, 0xde, 0x5e, 0x0b, 0xdb, 0xe0,
	0x32, 0x3a, 0x0a, 0x49, 0x06, 0x24, 0x5c, 0xc2, 0xd3, 0xac, 0x62, 0x91, 0x95, 0xe4, 0x79, 0xe7, 0xc8, 0x37, 0x6d, 0x8d, 0xd5, 0x4e, 0xa9,
	0x6c, 0x56, 0xf4, 0xea, 0x65, 0x7a, 0xae, 0x08, 0xba, 0x78, 0x25, 0x2e, 0x1c, 0xa6, 0xb4, 0xc6, 0xe8, 0xdd, 0x74, 0x1f, 0x4b, 0xbd, 0x8b,
	0x8a, 0x70, 0x3e, 0xb5, 0x66, 0x48, 0x03, 0xf6, 0x0e, 0x61, 0x35, 0x57, 0xb9, 0x86, 0xc1, 0x1d, 0x9e, 0xe1, 0xf8, 0x98, 0x11, 0x69, 0xd9,
	0x8e, 0x94, 0x9b, 0x1e, 0x87, 0xe9, 0xce, 0x55, 0x28, 0xdf, 0x8c, 0xa1, 0x89, 0x0d, 0xbf, 0xe6, 0x42, 0x68, 0x41, 0x99, 0x2d, 0x0f, 0xb0,
	0x54, 0xbb, 0x16};

__device__ __forceinline__ uint32_t aes_nk(uint32_t strength) { return 2u + 2u * strength; }   // key words: 4 / 6 / 8
__device__ __forceinline__ uint32_t aes_salt_len(uint32_t strength) { return 4u + 4u * strength; }
__device__ __forceinline__ uint32_t bswap32(uint32_t x) { return __byte_perm(x, 0, 0x0123); }
__device__ __forceinline__ uint32_t rotl32(uint32_t x, int n) { return __funnelshift_l(x, x, n); }

// ---------------------------------------------------------------- SHA-1 (FIPS 180-4), w[] is consumed
__device__ __forceinline__ void sha1_compress(uint32_t h[5], uint32_t w[16]) {
	uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4];
#pragma unroll
	for (int i = 0; i < 80; i++) {
		uint32_t wi;
		if (i < 16) {
			wi = w[i];
		} else {
			wi = rotl32(w[(i - 3) & 15] ^ w[(i - 8) & 15] ^ w[(i - 14) & 15] ^ w[i & 15], 1);
			w[i & 15] = wi;
		}
		uint32_t f, k;
		if (i < 20) {
			f = (b & c) | (~b & d);
			k = 0x5A827999u;
		} else if (i < 40) {
			f = b ^ c ^ d;
			k = 0x6ED9EBA1u;
		} else if (i < 60) {
			f = (b & c) | (b & d) | (c & d);
			k = 0x8F1BBCDCu;
		} else {
			f = b ^ c ^ d;
			k = 0xCA62C1D6u;
		}
		const uint32_t t = rotl32(a, 5) + f + e + k + wi;
		e = d;
		d = c;
		c = rotl32(b, 30);
		b = a;
		a = t;
	}
	h[0] += a;
	h[1] += b;
	h[2] += c;
	h[3] += d;
	h[4] += e;
}

__device__ __forceinline__ void sha1_init(uint32_t h[5]) {
	h[0] = 0x67452301u;
	h[1] = 0xEFCDAB89u;
	h[2] = 0x98BADCFEu;
	h[3] = 0x10325476u;
	h[4] = 0xC3D2E1F0u;
}

// One 64-byte block of p as big-endian words; bytes at or beyond `avail` read as zero, byte `avail` as the 0x80 pad
// marker when pad is set.
__device__ __forceinline__ void sha1_load(uint32_t w[16], const uint8_t *p, uint64_t avail, bool pad) {
	if (avail >= 64 && !((uintptr_t)p & 15)) {
#pragma unroll
		for (int j = 0; j < 4; j++) {
			const uint4 v = ld_stream16(p + 16 * j);
			w[4 * j + 0] = bswap32(v.x);
			w[4 * j + 1] = bswap32(v.y);
			w[4 * j + 2] = bswap32(v.z);
			w[4 * j + 3] = bswap32(v.w);
		}
		return;
	}
#pragma unroll
	for (int j = 0; j < 16; j++) {
		uint32_t x = 0;
#pragma unroll
		for (int q = 0; q < 4; q++) {
			const uint64_t i = 4 * j + q;
			const uint32_t b = i < avail ? p[i] : (pad && i == avail) ? 0x80u : 0u;
			x |= b << (24 - 8 * q);
		}
		w[j] = x;
	}
}

// Absorb len bytes of p and the final padding into h; `prefix` bytes were absorbed before (the HMAC key block).
__device__ __forceinline__ void sha1_tail(uint32_t h[5], const uint8_t *p, uint64_t len, uint64_t prefix) {
	uint32_t w[16];
	uint64_t o = 0;
	for (; len - o >= 64; o += 64) {
		sha1_load(w, p + o, 64, false);
		sha1_compress(h, w);
	}
	const uint64_t rem = len - o;
	sha1_load(w, p + o, rem, true);
	if (rem >= 56) {
		sha1_compress(h, w);
#pragma unroll
		for (int j = 0; j < 16; j++) {
			w[j] = 0;
		}
	}
	const uint64_t bits = (prefix + len) * 8;
	w[14] = (uint32_t)(bits >> 32);
	w[15] = (uint32_t)bits;
	sha1_compress(h, w);
}

// h = state after the 64-byte block (key ^ pad), key given as big-endian words (zero beyond its length)
__device__ __forceinline__ void hmac_key_state(uint32_t h[5], const uint32_t key[16], uint32_t pad) {
	uint32_t w[16];
#pragma unroll
	for (int j = 0; j < 16; j++) {
		w[j] = key[j] ^ pad;
	}
	sha1_init(h);
	sha1_compress(h, w);
}

// one HMAC over a 20-byte message u (in place): inner hash of u, outer hash of that
__device__ __forceinline__ void hmac20(uint32_t u[5], const uint32_t hi[5], const uint32_t ho[5]) {
	uint32_t w[16], s[5];
#pragma unroll
	for (int j = 0; j < 5; j++) {
		w[j] = u[j];
		s[j] = hi[j];
	}
	w[5] = 0x80000000u;
#pragma unroll
	for (int j = 6; j < 15; j++) {
		w[j] = 0;
	}
	w[15] = (64 + 20) * 8;
	sha1_compress(s, w);
#pragma unroll
	for (int j = 0; j < 5; j++) {
		w[j] = s[j];
		u[j] = ho[j];
	}
	w[5] = 0x80000000u;
#pragma unroll
	for (int j = 6; j < 15; j++) {
		w[j] = 0;
	}
	w[15] = (64 + 20) * 8;
	sha1_compress(u, w);
}

// ---------------------------------------------------------------- k_aes_kdf
// pw_bytes[pw_ofs[k] .. pw_ofs[k + 1]) is password k.  seal = 0: compare the verification value at pwv_base + job.pwv and
// set verdict[e] to OTZ_ST_OK / OTZ_ST_WRONGPASSWD (OTZ_ST_NOPASSWD without a password); seal = 1: write it there, and the
// salt to pwv_base + job.hdr.
__global__ void __launch_bounds__(OTZ_AES_KDF_THREADS) k_aes_kdf(const OtzAesJob *__restrict__ jobs, uint32_t n,
	const uint8_t *__restrict__ pw_bytes, const uint32_t *__restrict__ pw_ofs, uint32_t n_pw, const uint8_t *__restrict__ salt_base,
	uint8_t *__restrict__ pwv_base, uint64_t pwv_len, int seal, OtzAesKeys *__restrict__ keys, int32_t *__restrict__ verdict) {
	__shared__ uint32_t s_dk[OTZ_AES_KDF_THREADS / 4][20];
	__shared__ uint8_t s_sbox[256];
	for (int i = threadIdx.x; i < 256; i += blockDim.x) {
		s_sbox[i] = g_aes_sbox[i];
	}
	__syncthreads();
	const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t e = g >> 2, t = g & 3, le = threadIdx.x >> 2;
	const bool live = e < n;
	OtzAesJob jb;
	uint32_t nk = 4, nblk = 0;
	bool has_pw = false;
	if (live) {
		jb = jobs[e];
		nk = aes_nk(jb.strength);
		nblk = (2 * 4 * nk + 2 + 19) / 20;
		has_pw = jb.pw < n_pw;
	}
	if (live && has_pw && t < nblk) {
		// the HMAC key is the password, or its SHA-1 when it is longer than the block
		const uint8_t *pw = pw_bytes + pw_ofs[jb.pw];
		const uint32_t pl = pw_ofs[jb.pw + 1] - pw_ofs[jb.pw];
		uint32_t key[16];
		if (pl > 64) {
			uint32_t h[5];
			sha1_init(h);
			sha1_tail(h, pw, pl, 0);
#pragma unroll
			for (int j = 0; j < 16; j++) {
				key[j] = j < 5 ? h[j] : 0u;
			}
		} else {
			sha1_load(key, pw, pl, false);
		}
		uint32_t hi[5], ho[5];
		hmac_key_state(hi, key, 0x36363636u);
		hmac_key_state(ho, key, 0x5C5C5C5Cu);
		// U_1 = HMAC(salt || INT(t + 1))
		const uint32_t sl = aes_salt_len(jb.strength);
		uint32_t w[16];
		sha1_load(w, salt_base + jb.salt, sl, false);
		const uint32_t sw = sl / 4;
#pragma unroll
		for (int j = 0; j < 16; j++) {
			if (j == (int)sw) {
				w[j] = t + 1;
			} else if (j == (int)sw + 1) {
				w[j] = 0x80000000u;
			}
		}
		w[15] = (64 + sl + 4) * 8;
		uint32_t u[5];
#pragma unroll
		for (int j = 0; j < 5; j++) {
			u[j] = hi[j];
		}
		sha1_compress(u, w);
#pragma unroll
		for (int j = 0; j < 5; j++) {
			w[j] = u[j];
			u[j] = ho[j];
		}
		w[5] = 0x80000000u;
#pragma unroll
		for (int j = 6; j < 15; j++) {
			w[j] = 0;
		}
		w[15] = (64 + 20) * 8;
		sha1_compress(u, w);
		uint32_t acc[5];
#pragma unroll
		for (int j = 0; j < 5; j++) {
			acc[j] = u[j];
		}
		for (int it = 1; it < OTZ_AES_ITER; it++) {
			hmac20(u, hi, ho);
#pragma unroll
			for (int j = 0; j < 5; j++) {
				acc[j] ^= u[j];
			}
		}
#pragma unroll
		for (int j = 0; j < 5; j++) {
			s_dk[le][5 * t + j] = acc[j];
		}
	}
	__syncwarp();
	if (!live) {
		return;
	}
	const uint32_t *dk = s_dk[le];   // AES key | HMAC key | verification value, big-endian words
	if (t == 0) {
		int32_t v = OTZ_ST_OK;
		if (!has_pw) {
			v = OTZ_ST_NOPASSWD;
		} else {
			const uint32_t want = dk[2 * nk] >> 16;
			uint8_t *pv = pwv_base + jb.pwv;
			OTZ_CHK(jb.pwv + 2 <= pwv_len, seal ? OTZ_CK_AES_OUT : OTZ_CK_AES_IN);
			if (seal) {
				pv[0] = (uint8_t)(want >> 8);
				pv[1] = (uint8_t)want;
			} else if ((((uint32_t)pv[0] << 8) | pv[1]) != want) {
				v = OTZ_ST_WRONGPASSWD;
			}
		}
		verdict[e] = v;
		// FIPS-197 key expansion, straight into the entry's slot
		const uint32_t nr = nk + 6, nw = 4 * (nr + 1);
		uint32_t *rk = keys[e].rk;
		keys[e].nr = nr;
		uint32_t rcon = 1;
		for (uint32_t i = 0; i < nw; i++) {
			OTZ_CHK(i < 60, OTZ_CK_AES_RK);
			uint32_t x;
			if (i < nk) {
				x = has_pw ? dk[i] : 0u;
			} else {
				uint32_t tmp = rk[i - 1];
				if (i % nk == 0) {
					tmp = (tmp << 8) | (tmp >> 24);
					tmp = ((uint32_t)s_sbox[tmp >> 24] << 24) | ((uint32_t)s_sbox[(tmp >> 16) & 0xFF] << 16) |
						((uint32_t)s_sbox[(tmp >> 8) & 0xFF] << 8) | s_sbox[tmp & 0xFF];
					tmp ^= rcon << 24;
					rcon = (rcon << 1) ^ ((rcon & 0x80) ? 0x11Bu : 0u);
				} else if (nk > 6 && i % nk == 4) {
					tmp = ((uint32_t)s_sbox[tmp >> 24] << 24) | ((uint32_t)s_sbox[(tmp >> 16) & 0xFF] << 16) |
						((uint32_t)s_sbox[(tmp >> 8) & 0xFF] << 8) | s_sbox[tmp & 0xFF];
				}
				x = rk[i - nk] ^ tmp;
			}
			rk[i] = x;
		}
	} else if (t == 2 && seal) {
		const uint32_t sl = aes_salt_len(jb.strength);
		OTZ_CHK(jb.hdr + sl <= pwv_len, OTZ_CK_AES_OUT);
		for (uint32_t q = 0; q < sl; q++) {
			pwv_base[jb.hdr + q] = salt_base[jb.salt + q];
		}
	} else if (t == 1) {
		uint32_t key[16];
#pragma unroll
		for (int j = 0; j < 16; j++) {
			key[j] = 0;
		}
		for (uint32_t j = 0; j < nk && has_pw; j++) {
			const uint32_t x = dk[nk + j];
#pragma unroll
			for (int q = 0; q < 8; q++) {
				key[q] = (uint32_t)q == j ? x : key[q];
			}
		}
		uint32_t hs[5];
		hmac_key_state(hs, key, 0x36363636u);
#pragma unroll
		for (int j = 0; j < 5; j++) {
			keys[e].hi[j] = hs[j];
		}
		hmac_key_state(hs, key, 0x5C5C5C5Cu);
#pragma unroll
		for (int j = 0; j < 5; j++) {
			keys[e].ho[j] = hs[j];
		}
	}
}

// ---------------------------------------------------------------- k_aes_ctr
struct AesSmem {
	uint32_t te[4][256];
	uint32_t rk[60];
	uint8_t sbox[256];
};

__device__ __forceinline__ uint4 aes_keystream(const AesSmem &s, uint32_t nr, uint32_t ctr) {
	uint32_t s0 = bswap32(ctr) ^ s.rk[0], s1 = s.rk[1], s2 = s.rk[2], s3 = s.rk[3];
	for (uint32_t r = 1; r < nr; r++) {
		OTZ_CHK(4 * r + 3 < 60, OTZ_CK_AES_RK);
		const uint32_t t0 = s.te[0][s0 >> 24] ^ s.te[1][(s1 >> 16) & 0xFF] ^ s.te[2][(s2 >> 8) & 0xFF] ^ s.te[3][s3 & 0xFF] ^ s.rk[4 * r];
		const uint32_t t1 = s.te[0][s1 >> 24] ^ s.te[1][(s2 >> 16) & 0xFF] ^ s.te[2][(s3 >> 8) & 0xFF] ^ s.te[3][s0 & 0xFF] ^ s.rk[4 * r + 1];
		const uint32_t t2 = s.te[0][s2 >> 24] ^ s.te[1][(s3 >> 16) & 0xFF] ^ s.te[2][(s0 >> 8) & 0xFF] ^ s.te[3][s1 & 0xFF] ^ s.rk[4 * r + 2];
		const uint32_t t3 = s.te[0][s3 >> 24] ^ s.te[1][(s0 >> 16) & 0xFF] ^ s.te[2][(s1 >> 8) & 0xFF] ^ s.te[3][s2 & 0xFF] ^ s.rk[4 * r + 3];
		s0 = t0;
		s1 = t1;
		s2 = t2;
		s3 = t3;
	}
	OTZ_CHK(4 * nr + 3 < 60, OTZ_CK_AES_RK);
	const uint32_t *k = s.rk + 4 * nr;
	const uint8_t *sb = s.sbox;
	uint4 o;   // keystream as little-endian words, ready to XOR with 16-byte vector loads
	o.x = bswap32((((uint32_t)sb[s0 >> 24] << 24) | ((uint32_t)sb[(s1 >> 16) & 0xFF] << 16) | ((uint32_t)sb[(s2 >> 8) & 0xFF] << 8) | sb[s3 & 0xFF]) ^ k[0]);
	o.y = bswap32((((uint32_t)sb[s1 >> 24] << 24) | ((uint32_t)sb[(s2 >> 16) & 0xFF] << 16) | ((uint32_t)sb[(s3 >> 8) & 0xFF] << 8) | sb[s0 & 0xFF]) ^ k[1]);
	o.z = bswap32((((uint32_t)sb[s2 >> 24] << 24) | ((uint32_t)sb[(s3 >> 16) & 0xFF] << 16) | ((uint32_t)sb[(s0 >> 8) & 0xFF] << 8) | sb[s1 & 0xFF]) ^ k[2]);
	o.w = bswap32((((uint32_t)sb[s3 >> 24] << 24) | ((uint32_t)sb[(s0 >> 16) & 0xFF] << 16) | ((uint32_t)sb[(s1 >> 8) & 0xFF] << 8) | sb[s2 & 0xFF]) ^ k[3]);
	return o;
}

// hdr_image = 1 (open): the first chunk of every entry also writes the synthetic local header at job.hdr (signature, all
// other fields zero) — or a zeroed one when the entry's verification failed, so that its decode stops at the signature.
__global__ void __launch_bounds__(OTZ_AES_CTR_THREADS) k_aes_ctr(const OtzAesJob *__restrict__ jobs, uint32_t n,
	const OtzAesWork *__restrict__ work, uint32_t n_work, const OtzAesKeys *__restrict__ keys, const int32_t *__restrict__ verdict,
	const uint8_t *__restrict__ in, uint64_t in_len, uint8_t *__restrict__ out, uint64_t out_len, int hdr_image) {
	__shared__ AesSmem s;
	const uint32_t wi = blockIdx.x;
	OTZ_CHK(wi < n_work, OTZ_CK_AES_WORK);
	const OtzAesWork wk = work[wi];
	OTZ_CHK(wk.job < n, OTZ_CK_AES_WORK);
	const OtzAesJob jb = jobs[wk.job];
	const bool ok = verdict[wk.job] == OTZ_ST_OK;
	if (hdr_image && wk.chunk == 0 && threadIdx.x < 30) {
		OTZ_CHK(jb.hdr + 30 <= out_len, OTZ_CK_AES_OUT);
		const uint32_t sig = ok ? OTZ_SIG_LFH : 0u;
		out[jb.hdr + threadIdx.x] = threadIdx.x < 4 ? (uint8_t)(sig >> (8 * threadIdx.x)) : 0;
	}
	if (!ok) {
		return;
	}
	{
		const uint32_t x = threadIdx.x;
		const uint32_t sv = g_aes_sbox[x];
		const uint32_t s2 = ((sv << 1) ^ ((sv & 0x80) ? 0x1Bu : 0u)) & 0xFF, s3 = s2 ^ sv;
		const uint32_t t = (s2 << 24) | (sv << 16) | (sv << 8) | s3;
		OTZ_CHK(x < 256, OTZ_CK_AES_TAB);
		s.te[0][x] = t;
		s.te[1][x] = (t >> 8) | (t << 24);
		s.te[2][x] = (t >> 16) | (t << 16);
		s.te[3][x] = (t >> 24) | (t << 8);
		s.sbox[x] = (uint8_t)sv;
		if (x < 60) {
			s.rk[x] = keys[wk.job].rk[x];
		}
	}
	__syncthreads();
	const uint32_t nr = keys[wk.job].nr;
	const uint32_t nblk = (jb.len + 15) / 16;
	const uint32_t b0 = wk.chunk * (OTZ_AES_CHUNK / 16);
	const uint32_t b1 = min(nblk, b0 + OTZ_AES_CHUNK / 16);
	const uint8_t *src = in + jb.src;
	uint8_t *dst = out + jb.dst;
	const bool vec = !(((uintptr_t)src | (uintptr_t)dst) & 15);
	for (uint32_t b = b0 + threadIdx.x; b < b1; b += blockDim.x) {
		const uint4 k = aes_keystream(s, nr, b + 1);
		const uint64_t o = 16ull * b;
		const uint32_t m = jb.len - (uint32_t)o < 16u ? jb.len - (uint32_t)o : 16u;
		OTZ_CHK(jb.src + o + m <= in_len, OTZ_CK_AES_IN);
		OTZ_CHK(jb.dst + o + m <= out_len, OTZ_CK_AES_OUT);
		if (vec && m == 16) {
			uint4 v = ld_stream16(src + o);
			v.x ^= k.x;
			v.y ^= k.y;
			v.z ^= k.z;
			v.w ^= k.w;
			*reinterpret_cast<uint4 *>(dst + o) = v;
		} else {
			const uint32_t kw[4] = { k.x, k.y, k.z, k.w };
#pragma unroll
			for (uint32_t q = 0; q < 16; q++) {
				if (q < m) {
					dst[o + q] = src[o + q] ^ (uint8_t)(kw[q >> 2] >> (8 * (q & 3)));
				}
			}
		}
	}
}

// ---------------------------------------------------------------- k_aes_mac
// order[] lists the jobs longest first.  data + job.(seal ? dst : src) is the ciphertext.  Open: auth[e] = 1 when the
// stored code differs (only entries whose verification value matched are checked); seal: the code is written.
__global__ void k_aes_mac(const OtzAesJob *__restrict__ jobs, const uint32_t *__restrict__ order, uint32_t n,
	const OtzAesKeys *__restrict__ keys, const int32_t *__restrict__ verdict, const uint8_t *__restrict__ data, uint8_t *__restrict__ mac_base,
	uint64_t mac_len, int seal, int32_t *__restrict__ auth) {
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) {
		return;
	}
	const uint32_t e = order[i];
	OTZ_CHK(e < n, OTZ_CK_AES_WORK);
	const OtzAesJob jb = jobs[e];
	if (verdict[e] != OTZ_ST_OK) {
		auth[e] = 0;
		return;
	}
	uint32_t h[5], w[16];
#pragma unroll
	for (int j = 0; j < 5; j++) {
		h[j] = keys[e].hi[j];
	}
	OTZ_CHK((seal ? jb.dst : jb.src) + jb.len <= mac_len, OTZ_CK_AES_IN);   // (data and mac_base are the same buffer)
	sha1_tail(h, data + (seal ? jb.dst : jb.src), jb.len, 64);
	uint32_t m[5];
#pragma unroll
	for (int j = 0; j < 5; j++) {
		w[j] = h[j];
		m[j] = keys[e].ho[j];
	}
	w[5] = 0x80000000u;
#pragma unroll
	for (int j = 6; j < 15; j++) {
		w[j] = 0;
	}
	w[15] = (64 + 20) * 8;
	sha1_compress(m, w);
	uint8_t *mc = mac_base + jb.mac;
	OTZ_CHK(jb.mac + 10 <= mac_len, seal ? OTZ_CK_AES_OUT : OTZ_CK_AES_IN);
	uint32_t diff = 0;
#pragma unroll
	for (int q = 0; q < 10; q++) {
		const uint8_t b = (uint8_t)(m[q >> 2] >> (24 - 8 * (q & 3)));
		if (seal) {
			mc[q] = b;
		} else {
			diff |= (uint32_t)(mc[q] ^ b);   // constant time: every byte is compared
		}
	}
	auth[e] = diff != 0;
}

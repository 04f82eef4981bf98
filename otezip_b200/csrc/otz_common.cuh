// otz_common.cuh — shared device helpers for the otezip_b200 kernels (sm_100a).
#pragma once

#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/otz_gpu.h"

namespace cg = cooperative_groups;

// ---------------------------------------------------------------- software bounds checks (debug build)
// compute-sanitizer is not available on the GPU pool this was developed on, so the kernels written with unmasked /
// word-granular / per-lane indexed accesses carry their own checks: `make debug` builds libotezip_b200_dbg.so with
// -DOTZ_BOUNDS_CHECK, every OTZ_CHK site counts its violations in g_otz_violations[code], tests/test_gpu_bounds.py runs
// the parity suite's hardest cases against that build and requires all counters to be zero (otz_debug_violations).
// In the release build the macro compiles to nothing.
#define OTZ_CHK_SLOTS 31
#ifdef OTZ_BOUNDS_CHECK
__device__ unsigned long long g_otz_violations[OTZ_CHK_SLOTS];
#define OTZ_CHK(cond, code)                                     \
	do {                                                        \
		if (!(cond)) {                                          \
			atomicAdd(&g_otz_violations[(code)], 1ull);         \
		}                                                       \
	} while (0)
#else
#define OTZ_CHK(cond, code) \
	do {                    \
	} while (0)
#endif
// check sites
#define OTZ_CK_SPEC_PIECE 0     // k_inflate_spec: a decoding position left the words staged for its piece
#define OTZ_CK_SPEC_VIS 1       // k_inflate_spec: visited-bitmap index outside the piece
#define OTZ_CK_SPEC_LIT 2       // k_inflate_spec: literal store outside the stream's token scratch
#define OTZ_CK_SPEC_SEQ 3       // k_inflate_spec: record store outside the stream's token scratch / below the literals
#define OTZ_CK_SPEC_STORED 4    // k_inflate_spec: stored-block payload copy outside input or scratch
#define OTZ_CK_LZ_RING_DST 5    // k_inflate_lz: unmasked ring store outside the ring
#define OTZ_CK_LZ_RING_SRC 6    // k_inflate_lz: unmasked source load outside ring + staging buffers
#define OTZ_CK_LZ_STAGE 7       // k_inflate_lz: far source staged outside its staging buffer
#define OTZ_CK_LZ_FLUSH 9       // k_inflate_lz: ring flush outside the entry's slice of the arena / symbol buffer
#define OTZ_CK_SEG_TABLE 12     // k_inflate_spec: segment table index beyond I2_MAXSEG
#define OTZ_CK_ZS_TABLE 13      // k_zstd_seq: FSE state outside its table
#define OTZ_CK_ZS_REC 14        // k_zstd_seq: sequence record stored below the literals of the entry's token scratch
#define OTZ_CK_ZS_LIT 15        // k_zstd_lit: literals of a block outside the entry's token scratch
#define OTZ_CK_DFL_PAIR 16      // k_deflate_chunks: (token, way) pair of the second search pass outside the window / the chunk
#define OTZ_CK_AES_RK 17        // k_aes_kdf / k_aes_ctr: round-key word beyond the 60 of AES-256
#define OTZ_CK_AES_TAB 18       // k_aes_ctr: T-table / S-box slot beyond 256
#define OTZ_CK_AES_WORK 19      // k_aes_ctr / k_aes_mac: work-list or job index out of range
#define OTZ_CK_AES_OUT 20       // k_aes_ctr: plaintext-image / ciphertext store outside the output buffer
#define OTZ_CK_AES_IN 21        // k_aes_ctr: load outside the input buffer
#define OTZ_CK_D64_OUT 22       // k_inflate<D64>: piece of a long match beyond the entry's output slice
#define OTZ_CK_D64_SRC 23       // k_inflate<D64>: piece source neither in the ring nor flushed to HBM, or before the slice
#define OTZ_CK_DFB_LINK 24      // k_deflate_best: hash-chain link that is not an earlier position of the chunk
#define OTZ_CK_DFB_STAGE 25     // k_deflate_best: word read beyond the staged chunk
#define OTZ_CK_DFB_STORE 26     // k_deflate_best: match-table / token store outside the slot, or ahead of the parse
#define OTZ_CK_XZ_SEG 27        // k_xz_walk: segment beyond the entry's slot range of the segment table
#define OTZ_CK_XZ_IN 28         // k_lzma: uncompressed-chunk load beyond the entry's payload
#define OTZ_CK_XZ_PROB 29       // k_lzma: probability index beyond the model of the segment's class
#define OTZ_CK_XZ_OUT 30        // k_lzma: output store beyond the segment's part of the entry's slice

#define OTZ_SIG_LFH 0x04034b50u
#define OTZ_MAX_PAYLOAD (2ull * 1024ull * 1024ull * 1024ull)  // otezip.c:102

// Per-entry device state produced by k_resolve and consumed by the decoders.
struct OtzEntryState {
	uint64_t data_ofs;   // offset of the compressed payload in the archive image
};

// ---------------------------------------------------------------- unaligned little-endian reads
__device__ __forceinline__ uint32_t ld_u8(const uint8_t *p) { return *p; }
__device__ __forceinline__ uint32_t ld_le16(const uint8_t *p) { return p[0] | (p[1] << 8); }
__device__ __forceinline__ uint32_t ld_le32(const uint8_t *p) {
	return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24);
}

// 16-byte streaming load (read-once data: keep it out of L1)
__device__ __forceinline__ uint4 ld_stream16(const void *p) {
	uint4 r;
	asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
		: "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
	return r;
}
__device__ __forceinline__ void st_stream16(void *p, uint4 v) {
	asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---------------------------------------------------------------- CRC-32 polynomial arithmetic
// Reflected representation, as crc32.inc.c:40-47 uses it: bit 31 is x^0.
#define OTZ_CRC_POLY 0xEDB88320u

// a(x) * b(x) mod P(x)
__device__ __forceinline__ uint32_t crc_mulmod(uint32_t a, uint32_t b) {
	uint32_t p = 0;
#pragma unroll
	for (int i = 0; i < 32; i++) {
		p ^= (a & (0x80000000u >> i)) ? b : 0u;
		b = (b >> 1) ^ ((b & 1u) ? OTZ_CRC_POLY : 0u);
	}
	return p;
}

// Tables resident in global memory (filled once per context by the host).
struct OtzCrcTables {
	uint32_t skip[16][256];   // skip[i][b]: CRC state contribution of byte b followed by 511-i zero bytes
	uint32_t x2n[32];         // x^(2^k) mod P
	uint32_t xp8[1024 + 64];  // xp8[k + OTZ_XP8_BIAS] = x^(8k) mod P for k in [-OTZ_XP8_BIAS, 1024+64-BIAS)
	uint32_t t0[256];         // plain byte table
	uint32_t x_inv_fold;      // x^(-8 * 512 * FOLD_K): undoes the zero rows the fold path appends
};
#define OTZ_XP8_BIAS 528

// x^(8*n) mod P for arbitrary byte counts (serial square-and-multiply over the bits of n).
__device__ __forceinline__ uint32_t crc_xpow8(uint64_t nbytes, const uint32_t *__restrict__ x2n) {
	uint32_t p = 0x80000000u;  // x^0
	int k = 3;                 // x^(2^3) = x^8
	while (nbytes) {
		if (nbytes & 1) {
			p = crc_mulmod(x2n[k & 31], p);
		}
		nbytes >>= 1;
		k++;
	}
	return p;
}

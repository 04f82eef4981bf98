// k_deflate_best.cuh — phase 1 (LZ77) of the best DEFLATE level (libzip levels 7-9, OTZ_M_BEST), one CTA per chunk.
//
// The chunk contract is the one of k_deflate_chunks: 65,280-byte chunks, matches inside the chunk and within 32,768 bytes,
// one dynamic block (or a stored one) closed by an empty stored block, so every chunk is byte-aligned and decodes on its
// own.  Only the match search and the parse differ; phases 2 and 3 are dfl_code_emit (k_deflate.cuh).
//
// Per chunk (scheme and parameters from tools/dfl_parse_sim.c `best`: ratio 9.91 on the c5 corpus, zlib level 6 on
// whole entries 9.38):
//  (1) the chunk is staged in shared memory as words;
//  (2) one warp links every position into hash chains (4-byte hash, 2^14 heads, prev[] of 16-bit links, both in shared
//      memory): 32 positions per step, lanes with equal hash linked in position order through __match_any_sync, so the
//      chains are exactly the serial ones;
//  (3) every position is searched on its own by all threads of the CTA: the chain is walked to DFB_CHAIN links, a
//      candidate that cannot beat the current match is dropped after one 4-byte comparison (zlib's scan_end test), a
//      longer match wins and the nearer one on equal lengths, and only a match that cannot grow (258 bytes or the chunk
//      end: nice length 258) ends the walk early.  Each position's match goes to the token slot as a token;
//  (4) one warp parses the per-position matches with the two-step lazy rule (a match is taken unless the next position
//      has a longer one or the one after that a match longer by two), rewriting the slot into the token array in place
//      (a token never overtakes the positions still to be read), with the symbol histograms for phase 2.
// Every step is a pure function of the chunk's bytes: the output does not depend on the grid or on timing.
#pragma once
#include "k_deflate.cuh"

#define DFB_THREADS 512
#define DFB_HASH_BITS 14                        // 2^14 chain heads of 16 bits: 32 KiB
#define DFB_CHAIN 128                           // chain links walked per position (zlib level 9: 4,096; the model: 9.91 vs 10.01)
#define DFB_STAGE_WORDS (DFL_CHUNK / 4 + 4)     // the chunk plus zero words that the last word-wise comparisons read
#define DFB_SMEM (DFB_STAGE_WORDS * 4 + (1u << DFB_HASH_BITS) * 2 + DFL_CHUNK * 2)
static_assert(sizeof(DeflateSmem) <= DFL_CHUNK * 2, "phases 2/3 reuse the chain links' space");
static_assert(DFB_SMEM <= 227 * 1024, "shared memory of one CTA");

// unaligned 32-bit read of staged bytes [x, x + 4)
__device__ __forceinline__ uint32_t dfb_word(const uint32_t *s, uint32_t x) {
	const uint32_t i = x >> 2;
	OTZ_CHK(i + 1 < DFB_STAGE_WORDS, OTZ_CK_DFB_STAGE);
	return __funnelshift_r(s[i], s[i + 1], (x & 3u) * 8u);
}

// common prefix of the staged strings at c < p, at most maxl bytes
__device__ __forceinline__ uint32_t dfb_extend(const uint32_t *s, uint32_t c, uint32_t p, uint32_t maxl) {
	uint32_t l = 0;
	while (l < maxl) {
		const uint32_t x = dfb_word(s, c + l) ^ dfb_word(s, p + l);
		if (x) {
			l += (__ffs(x) - 1) >> 3;
			break;
		}
		l += 4;
	}
	return min(l, maxl);
}

// grid: persistent, sized by the occupancy of this kernel; chunks [first, first + n) of `chunks`, handed out in order.
// tokens: one DFL_CHUNK-word slot per CTA.
__global__ void __launch_bounds__(DFB_THREADS, 1) k_deflate_best(const uint8_t *__restrict__ in, const OtzDflChunk *__restrict__ chunks,
	uint32_t first, uint32_t n_best, uint32_t *__restrict__ tokens, uint8_t *__restrict__ cout, uint32_t *__restrict__ csize,
	uint32_t *__restrict__ work_counter) {
	extern __shared__ __align__(16) uint8_t smem_raw[];
	__shared__ uint32_t s_ci;
	uint32_t *stage = reinterpret_cast<uint32_t *>(smem_raw);
	uint16_t *head = reinterpret_cast<uint16_t *>(smem_raw + DFB_STAGE_WORDS * 4);
	uint16_t *prev = head + (1u << DFB_HASH_BITS);   // position + 1 of the previous position with the same hash, 0 = none
	DeflateSmem &S = *reinterpret_cast<DeflateSmem *>(prev);   // phases 2/3, once the search is done
	const uint32_t tid = threadIdx.x;
	const int lane = tid & 31;
	const bool warp0 = tid < 32;
	uint32_t *tok = tokens + (uint64_t)blockIdx.x * DFL_CHUNK;
	for (;;) {
		if (tid == 0) {
			s_ci = atomicAdd(work_counter, 1u);
		}
		__syncthreads();
		const uint32_t k = s_ci;
		if (k >= n_best) {
			break;
		}
		const uint32_t ci = first + k;
		const OtzDflChunk ck = chunks[ci];
		const uint32_t n = ck.len;
		const uint64_t ia = reinterpret_cast<uint64_t>(in + ck.in_ofs);
		const uint32_t *w = reinterpret_cast<const uint32_t *>(ia & ~3ull);
		const uint32_t sh0 = (uint32_t)(ia & 3ull);

		// ---- (1) stage the chunk, clear the heads
		for (uint32_t i = tid; i < DFB_STAGE_WORDS; i += DFB_THREADS) {
			uint32_t v = 0;
			if (4 * i < n) {
				v = dfl_word(w, sh0 + 4 * i);
				if (n - 4 * i < 4) {
					v &= (1u << (8 * (n - 4 * i))) - 1u;
				}
			}
			stage[i] = v;
		}
		for (uint32_t i = tid; i < (1u << DFB_HASH_BITS) / 2; i += DFB_THREADS) {
			reinterpret_cast<uint32_t *>(head)[i] = 0;
		}
		__syncthreads();

		// ---- (2) hash chains, one warp
		if (warp0) {
			for (uint32_t base = 0; base < n; base += 32) {
				const uint32_t p = base + lane;
				const bool can = p + DFL_MIN_MATCH <= n;
				uint32_t h = 0xFFFFFFFFu, old = 0;
				if (can) {
					h = (dfb_word(stage, p) * 2654435761u) >> (32 - DFB_HASH_BITS);
					old = head[h];
				}
				const uint32_t same = __match_any_sync(0xFFFFFFFFu, h);
				if (can) {
					const uint32_t lower = same & ((1u << lane) - 1u);   // earlier lanes of this step with the same hash
					const uint32_t link = lower ? base + 32u - __clz(lower) : old;   // (the nearest one, as position + 1)
					OTZ_CHK(p < DFL_CHUNK && link <= p, OTZ_CK_DFB_LINK);
					prev[p] = (uint16_t)link;
					if (lane == 31 - __clz(same)) {
						head[h] = (uint16_t)(p + 1u);
					}
				}
			}
		}
		__syncthreads();

		// ---- (3) the longest match of every position
		for (uint32_t p = tid; p < n; p += DFB_THREADS) {
			uint32_t rec = 0;
			if (p + DFL_MIN_MATCH <= n) {
				const uint32_t maxl = min((uint32_t)DFL_MAX_MATCH, n - p);
				uint32_t best = DFL_MIN_MATCH - 1, bd = 0;
				uint32_t c = prev[p];
				for (int d = 0; d < DFB_CHAIN && c; d++) {
					const uint32_t cp = c - 1u;
					OTZ_CHK(cp < p, OTZ_CK_DFB_LINK);
					if (p - cp > 32768u) {   // RFC 1951 window; the chain only gets older
						break;
					}
					// bytes [best - 3, best + 1): equal for every candidate that matches best + 1 bytes
					if (dfb_word(stage, cp + best - 3u) == dfb_word(stage, p + best - 3u)) {
						const uint32_t l = dfb_extend(stage, cp, p, maxl);
						if (l > best) {
							best = l;
							bd = p - cp;
							if (l == maxl) {
								break;
							}
						}
					}
					c = prev[cp];
				}
				if (bd) {
					rec = 0x80000000u | ((bd - 1u) << 8) | (best - 3u);
				}
			}
			OTZ_CHK(p < DFL_CHUNK, OTZ_CK_DFB_STORE);
			tok[p] = rec;
		}
		__syncthreads();
		if (!warp0) {
			continue;
		}

		// ---- (4) lazy parse, one warp; the match table becomes the token array in place
		for (int i = lane; i < 288; i += 32) {
			S.hist_ll[i] = 0;
		}
		S.hist_d[lane] = 0;
		if (lane < 4) {
			S.misc[lane] = 0;
		}
		__syncwarp();
		uint32_t ntok = 0, cur = 0;
		while (cur < n) {
			const uint32_t a = cur + lane < n ? tok[cur + lane] : 0u;
			const uint32_t b = (lane < 2 && cur + 32 + lane < n) ? tok[cur + 32 + lane] : 0u;
			const uint32_t la = a ? (a & 0xFFu) + 3u : 0u, lb = b ? (b & 0xFFu) + 3u : 0u;
			uint32_t i = 0, t = 0, mytok = 0;
			const uint32_t lim = min(32u, n - cur);
			while (i < lim) {
				const uint32_t L = __shfl_sync(0xFFFFFFFFu, la, i);
				const uint32_t Ln = __shfl_sync(0xFFFFFFFFu, i + 1 < 32 ? la : lb, (i + 1) & 31);
				const uint32_t Ln2 = __shfl_sync(0xFFFFFFFFu, i + 2 < 32 ? la : lb, (i + 2) & 31);
				const uint32_t m = __shfl_sync(0xFFFFFFFFu, a, i);
				uint32_t tokv;
				if (L && Ln <= L && Ln2 <= L + 1u) {
					tokv = m;
					i += L;
				} else {
					tokv = 0x40000000u | i;   // literal of window position i
					i += 1;
				}
				if ((uint32_t)lane == t) {
					mytok = tokv;
				}
				t++;
			}
			if ((uint32_t)lane < t) {
				if (mytok & 0x80000000u) {
					uint32_t xb, xv;
					const uint32_t ls = dfl_len_sym(mytok & 0xFFu, xb, xv);
					atomicAdd(&S.hist_ll[ls], 1u);
					uint32_t xb2;
					const uint32_t ds = dfl_dist_sym((mytok >> 8) & 0x7FFFu, xb2, xv);
					atomicAdd(&S.hist_d[ds], 1u);
					atomicAdd(&S.misc[0], xb + xb2);
				} else {
					const uint32_t x = cur + (mytok & 31u);
					mytok = (stage[x >> 2] >> ((x & 3u) * 8u)) & 0xFFu;
					atomicAdd(&S.hist_ll[mytok], 1u);
				}
				OTZ_CHK(ntok + lane < cur + i && ntok + lane < DFL_CHUNK, OTZ_CK_DFB_STORE);
				tok[ntok + lane] = mytok;
			}
			ntok += t;
			cur += i;
		}
		__syncwarp();
		dfl_code_emit(S, tok, ntok, in, ck, cout + (uint64_t)ci * DFL_OUT_STRIDE, csize, ci);
	}
}

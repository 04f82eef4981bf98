// k_deflate.cuh — batched raw-DEFLATE compressor, one warp per <=65,280-byte chunk of a source.
//
// Replaces otezip_compress_data's DEFLATE arm and deflateInit2/deflate/deflateEnd
// (/root/reference/src/lib/otezip.c:817-852; src/lib/deflate-enc.inc.c:199-541, "enc" below).
// The reference emits ONE fixed-Huffman block with a single-candidate greedy matcher and — because
// it writes its codes without bit reversal (enc:186-188 vs enc:157-183) and matches against bytes it
// has not written yet (enc:82-92) — produces streams nothing can decode (SURVEY.md F2).  Its behaviour
// is therefore replaced, not matched; what is kept is the caller contract: raw stream, STORE fallback
// when out >= in (otezip.c:846-850), zero-length -> STORE (otezip.c:793-801).
//
// Stream shape: every chunk becomes one dynamic-Huffman block (or one stored block when that is
// smaller) followed by an empty stored block, so every chunk starts and ends on a byte boundary and
// chunk outputs concatenate with memcpy; matches never cross a chunk start, so each chunk is also
// independently decodable.  The empty stored block of the last chunk carries BFINAL=1, which is the
// tail the reference's inflater always accepts (its end-of-input rule, SURVEY.md F1 / dec:811-816).
//
// Per chunk, one warp: (1) LZ77 — 32 consecutive positions per step, one per lane: 4-byte hash,
// single most-recent candidate from a 4096-entry shared-memory table, word-wise match extension,
// greedy parse with one-step lazy evaluation by shuffles; tokens and symbol histograms go to
// scratch / shared memory; (2) length-limited canonical Huffman codes (in-place minimum-redundancy
// construction on rank-sorted frequencies, lane 0) and the RLE-coded header; (3) 32 tokens per step
// are turned into bit strings, prefix-summed and OR-ed into a shared staging window that is flushed
// to the chunk's output with coalesced word stores.
#pragma once
#include "otz_common.cuh"
#include "k_copy.cuh"
#include "k_zstd_enc.cuh"

#define DFL_CHUNK 65280u                      // <= 65535 so the stored fallback is one block
#define DFL_OUT_STRIDE (DFL_CHUNK + 256u)     // per-chunk output slot (4-byte aligned)
#define DFL_HASH_BITS 12                      // 16-bit slots of the hash table: 8 KiB per chunk
#define DFL_WAYS 8                            // slots per bucket: the last eight positions with the same hash
#define DFL_BUCKET_BITS 9                     // 512 buckets (DFL_HASH_BITS - log2(DFL_WAYS))
#define DFL_MIN_MATCH 4
#define DFL_MAX_MATCH 258

struct OtzDflChunk {
	uint64_t in_ofs;     // absolute offset of the chunk in the input buffer
	uint32_t len;
	uint32_t entry;
	uint32_t last;       // bit 0: last chunk of its entry, bit 1: first chunk, bit 2: method 93 (Zstandard block instead of DEFLATE), bit 3: fast (first match pass only)
	uint32_t pad;        // length of the whole entry (Frame_Content_Size of a Zstandard frame)
};

struct __align__(16) DeflateSmem {
	union {
		uint16_t ht[1 << DFL_HASH_BITS];          // phase 1
		struct {                                  // phases 2/3
			uint32_t A[288];
			uint16_t order[288];
			uint8_t clens[320];
			uint8_t rle[320 * 2];
			// (the codes and the staging window are phase 2/3 as well: they share the hash table's space, which
			// makes room for a seventh CTA per SM)
			uint16_t code_ll[288];
			uint16_t code_d[32];
			uint8_t len_ll[288];
			uint8_t len_d[32];
			uint32_t hist_cl[19];
			uint16_t code_cl[19];
			uint8_t len_cl[19];
			uint32_t stage[72];
		} b;
	} u;
	uint32_t hist_ll[288];
	uint32_t hist_d[32];
	uint32_t misc[4];   // [0] extra-bit total of the chunk, [1] final byte count
	uint32_t best[32];  // phase 1, second pass: best (length << 16 | 32768 - distance) found for window position i
};

__device__ __forceinline__ uint32_t dfl_len_sym(uint32_t v /* len-3 */, uint32_t &xb, uint32_t &xv) {
	if (v < 8) {
		xb = 0;
		xv = 0;
		return 257 + v;
	}
	if (v == 255) {
		xb = 0;
		xv = 0;
		return 285;
	}
	const uint32_t e = 29 - __clz(v);
	xb = e;
	xv = v & ((1u << e) - 1u);
	return 257 + 4 * e + 4 + ((v >> e) & 3u);
}
__device__ __forceinline__ uint32_t dfl_dist_sym(uint32_t w /* dist-1 */, uint32_t &xb, uint32_t &xv) {
	if (w < 4) {
		xb = 0;
		xv = 0;
		return w;
	}
	const uint32_t e = 30 - __clz(w);
	xb = e;
	xv = w & ((1u << e) - 1u);
	return 2 * e + 2 + ((w >> e) & 1u);
}

// Unaligned 32-bit read at byte position x of a 4-byte aligned word array (may read one word past x).
__device__ __forceinline__ uint32_t dfl_word(const uint32_t *__restrict__ w, uint32_t x) {
	const uint32_t i = x >> 2, sh = (x & 3u) * 8u;
	return __funnelshift_r(__ldg(w + i), __ldg(w + i + 1), sh);
}

// ---- serial bit writer used by lane 0 for headers / trailers; continues the warp-level cursor
struct DflBits {
	uint32_t *out;     // chunk output as words
	uint64_t acc;
	uint32_t nacc;     // bits in acc (< 32 between calls)
	uint32_t wpos;     // next word index
	__device__ __forceinline__ void put(uint32_t v, uint32_t n) {
		acc |= (uint64_t)v << nacc;
		nacc += n;
		if (nacc >= 32) {
			out[wpos++] = (uint32_t)acc;
			acc >>= 32;
			nacc -= 32;
		}
	}
};

// In-place minimum-redundancy code lengths (Moffat & Katajainen) on ascending frequencies A[0..n).
__device__ __forceinline__ void dfl_min_redundancy(uint32_t *A, int n) {
	if (n == 1) {
		A[0] = 1;
		return;
	}
	A[0] += A[1];
	int root = 0, leaf = 2, next;
	for (next = 1; next < n - 1; next++) {
		if (leaf >= n || A[root] < A[leaf]) {
			A[next] = A[root];
			A[root++] = next;
		} else {
			A[next] = A[leaf++];
		}
		if (leaf >= n || (root < next && A[root] < A[leaf])) {
			A[next] += A[root];
			A[root++] = next;
		} else {
			A[next] += A[leaf++];
		}
	}
	A[n - 2] = 0;
	for (next = n - 3; next >= 0; next--) {
		A[next] = A[A[next]] + 1;
	}
	int avbl = 1, used = 0, dpth = 0;
	root = n - 2;
	next = n - 1;
	while (avbl > 0) {
		while (root >= 0 && (int)A[root] == dpth) {
			used++;
			root--;
		}
		while (avbl > used) {
			A[next--] = dpth;
			avbl--;
		}
		avbl = 2 * used;
		dpth++;
		used = 0;
	}
}

// Canonical, length-limited Huffman code for `nsym` symbols with frequencies hist[]; at least two symbols
// get a code (zlib does the same so that every decoder sees a complete set).  Whole warp; results in
// len_out[]/code_out[] (codes already bit-reversed for LSB-first emission).
__device__ __noinline__ void dfl_build_code(DeflateSmem &S, uint32_t *hist, int nsym, int maxbits, uint8_t *len_out, uint16_t *code_out) {
	const int lane = threadIdx.x & 31;
	if (lane == 0) {
		int nz = 0;
		for (int s = 0; s < nsym; s++) {
			nz += hist[s] != 0;
		}
		for (int s = 0; nz < 2 && s < nsym; s++) {
			if (hist[s] == 0) {
				hist[s] = 1;
				nz++;
			}
		}
	}
	__syncwarp();
	// rank sort of the used symbols by (frequency, symbol)
	int n = 0;
	for (int s = lane; s < nsym; s += 32) {
		const uint32_t f = hist[s];
		len_out[s] = 0;
		if (f) {
			int r = 0;
			for (int t = 0; t < nsym; t++) {
				const uint32_t g = hist[t];
				r += (g != 0) && (g < f || (g == f && t < s));
			}
			S.u.b.order[r] = (uint16_t)s;
			S.u.b.A[r] = f;
		}
	}
	for (int s = lane; s < nsym; s += 32) {
		n += hist[s] != 0;
	}
	for (int o = 16; o > 0; o >>= 1) {
		n += __shfl_xor_sync(0xFFFFFFFFu, n, o);
	}
	__syncwarp();
	if (lane == 0) {
		uint32_t *A = S.u.b.A;
		dfl_min_redundancy(A, n);
		// enforce the length limit (Kraft repair)
		int num[33];
		for (int i = 0; i <= 32; i++) {
			num[i] = 0;
		}
		for (int i = 0; i < n; i++) {
			num[A[i] > 32 ? 32 : A[i]]++;
		}
		for (int i = maxbits + 1; i <= 32; i++) {
			num[maxbits] += num[i];
		}
		uint32_t total = 0;
		for (int i = maxbits; i > 0; i--) {
			total += (uint32_t)num[i] << (maxbits - i);
		}
		while (total != (1u << maxbits)) {
			num[maxbits]--;
			for (int i = maxbits - 1; i > 0; i--) {
				if (num[i]) {
					num[i]--;
					num[i + 1] += 2;
					break;
				}
			}
			total--;
		}
		// least frequent symbols take the longest codes
		int k = 0;
		for (int l = maxbits; l >= 1; l--) {
			for (int c = 0; c < num[l]; c++) {
				len_out[S.u.b.order[k++]] = (uint8_t)l;
			}
		}
		// canonical codes, RFC 1951 3.2.2
		uint32_t next_code[17];
		uint32_t code = 0;
		next_code[0] = 0;
		for (int l = 1; l <= maxbits; l++) {
			code = (code + (uint32_t)num[l - 1] * (l > 1)) << 1;
			next_code[l] = code;
		}
		for (int s = 0; s < nsym; s++) {
			const int l = len_out[s];
			if (l) {
				code_out[s] = (uint16_t)(__brev(next_code[l]++) >> (32 - l));
			}
		}
	}
	__syncwarp();
}

// length of the common prefix of the strings at chunk positions c < p, at most maxl: 16 bytes per trip
__device__ __forceinline__ uint32_t dfl_extend(const uint32_t *__restrict__ w, uint32_t sh0, uint32_t c, uint32_t p, uint32_t maxl) {
	uint32_t l = 0;
	while (l < maxl) {
		const uint32_t ca = sh0 + c + l, pa = sh0 + p + l;
		const uint32_t ci = ca >> 2, cs = (ca & 3u) * 8u, pi = pa >> 2, ps = (pa & 3u) * 8u;
		const uint32_t c0 = __ldg(w + ci), c1 = __ldg(w + ci + 1), c2 = __ldg(w + ci + 2), c3 = __ldg(w + ci + 3), c4 = __ldg(w + ci + 4);
		const uint32_t p0 = __ldg(w + pi), p1 = __ldg(w + pi + 1), p2 = __ldg(w + pi + 2), p3 = __ldg(w + pi + 3), p4 = __ldg(w + pi + 4);
		const uint32_t x0 = __funnelshift_r(c0, c1, cs) ^ __funnelshift_r(p0, p1, ps);
		const uint32_t x1 = __funnelshift_r(c1, c2, cs) ^ __funnelshift_r(p1, p2, ps);
		const uint32_t x2 = __funnelshift_r(c2, c3, cs) ^ __funnelshift_r(p2, p3, ps);
		const uint32_t x3 = __funnelshift_r(c3, c4, cs) ^ __funnelshift_r(p3, p4, ps);
		if (x0 | x1) {
			l += x0 ? (__ffs(x0) - 1) >> 3 : 4 + ((__ffs(x1) - 1) >> 3);
			break;
		}
		if (x2 | x3) {
			l += x2 ? 8 + ((__ffs(x2) - 1) >> 3) : 12 + ((__ffs(x3) - 1) >> 3);
			break;
		}
		l += 16;
	}
	return min(l, maxl);
}

// Phases 2 and 3 of a DEFLATE chunk, one warp: Huffman codes from the histograms and the extra-bit total (S.misc[0]) that
// phase 1 left in S, the dynamic-block header, the stored-block fallback when that is not larger, and the emission of the
// ntok tokens of tok[] (a literal is the byte, a match 0x80000000 | (dist - 1) << 8 | (len - 3)) of chunk ci = ck into
// its output slot co; csize[ci] = bytes written.  k_deflate_chunks and k_deflate_best share it.
__device__ __forceinline__ void dfl_code_emit(DeflateSmem &S, const uint32_t *tok, uint32_t ntok, const uint8_t *in, const OtzDflChunk &ck,
	uint8_t *co, uint32_t *csize, uint32_t ci) {
	const int lane = threadIdx.x & 31;
	const uint32_t n = ck.len;
	const uint32_t xbits = S.misc[0];
	if (lane == 0) {
		S.hist_ll[256] = 1;   // end of block
	}
	__syncwarp();

	// ---------------- phase 2: Huffman codes + header cost
	dfl_build_code(S, S.hist_ll, 286, 15, S.u.b.len_ll, S.u.b.code_ll);
	dfl_build_code(S, S.hist_d, 30, 15, S.u.b.len_d, S.u.b.code_d);
	// code-length sequence with zero-run RLE (symbols 17/18), then the precode
	uint32_t hlit = 286, hdist = 30, nrle = 0;
	if (lane == 0) {
		while (hlit > 257 && S.u.b.len_ll[hlit - 1] == 0) {
			hlit--;
		}
		while (hdist > 1 && S.u.b.len_d[hdist - 1] == 0) {
			hdist--;
		}
		uint8_t *cl = S.u.b.clens;
		for (uint32_t i = 0; i < hlit; i++) {
			cl[i] = S.u.b.len_ll[i];
		}
		for (uint32_t i = 0; i < hdist; i++) {
			cl[hlit + i] = S.u.b.len_d[i];
		}
		for (int i = 0; i < 19; i++) {
			S.u.b.hist_cl[i] = 0;
		}
		const uint32_t tot = hlit + hdist;
		uint8_t *rle = S.u.b.rle;   // pairs (symbol, extra value)
		for (uint32_t i = 0; i < tot;) {
			if (cl[i] == 0) {
				uint32_t run = 1;
				while (i + run < tot && cl[i + run] == 0 && run < 138) {
					run++;
				}
				if (run >= 11) {
					rle[2 * nrle] = 18;
					rle[2 * nrle + 1] = (uint8_t)(run - 11);
					S.u.b.hist_cl[18]++;
					nrle++;
					i += run;
					continue;
				}
				if (run >= 3) {
					rle[2 * nrle] = 17;
					rle[2 * nrle + 1] = (uint8_t)(run - 3);
					S.u.b.hist_cl[17]++;
					nrle++;
					i += run;
					continue;
				}
			}
			rle[2 * nrle] = cl[i];
			rle[2 * nrle + 1] = 0;
			S.u.b.hist_cl[cl[i]]++;
			nrle++;
			i++;
		}
	}
	hlit = __shfl_sync(0xFFFFFFFFu, hlit, 0);
	hdist = __shfl_sync(0xFFFFFFFFu, hdist, 0);
	nrle = __shfl_sync(0xFFFFFFFFu, nrle, 0);
	__syncwarp();
	// the precode build reuses S.u.b.A/order: keep the RLE list (it lives in u.b.rle/clens)
	dfl_build_code(S, S.u.b.hist_cl, 19, 7, S.u.b.len_cl, S.u.b.code_cl);
	// exact size of the dynamic block
	uint32_t bits = 0;
	for (int s = lane; s < 286; s += 32) {
		bits += S.hist_ll[s] * S.u.b.len_ll[s];
	}
	if (lane < 30) {
		bits += S.hist_d[lane] * S.u.b.len_d[lane];
	}
	if (lane < 19) {
		bits += S.u.b.hist_cl[lane] * S.u.b.len_cl[lane] + (lane == 17 ? 3 * S.u.b.hist_cl[17] : lane == 18 ? 7 * S.u.b.hist_cl[18] : 0);
	}
	for (int o = 16; o > 0; o >>= 1) {
		bits += __shfl_xor_sync(0xFFFFFFFFu, bits, o);
	}
	bits += xbits + 3 + 14 + 19 * 3;
	const uint32_t dyn_bytes = (bits + 3 + 7) / 8 + 4;   // + empty stored block (3 bits, pad, LEN/NLEN)
	const uint32_t stored_bytes = 5 + n;
	uint32_t out_bytes;
	if (dyn_bytes >= stored_bytes) {
		// ---------------- stored block: [BFINAL|00 padded][LEN][NLEN][bytes]
		if (lane == 0) {
			co[0] = (uint8_t)(ck.last & 1u);
			co[1] = (uint8_t)(n & 0xFF);
			co[2] = (uint8_t)(n >> 8);
			co[3] = (uint8_t)(~n & 0xFF);
			co[4] = (uint8_t)((~n >> 8) & 0xFF);
		}
		tile_copy<32>(co + 5, in + ck.in_ofs, n, lane);
		out_bytes = stored_bytes;
	} else {
		// ---------------- phase 3: emit
		DflBits bw;
		bw.out = reinterpret_cast<uint32_t *>(co);
		bw.acc = 0;
		bw.nacc = 0;
		bw.wpos = 0;
		if (lane == 0) {
			bw.put(0u | (2u << 1), 3);   // BFINAL=0, BTYPE=10
			bw.put(hlit - 257, 5);
			bw.put(hdist - 1, 5);
			bw.put(19 - 4, 4);
			for (int i = 0; i < 19; i++) {
				bw.put(S.u.b.len_cl[c_cl_order[i]], 3);
			}
			const uint8_t *rle = S.u.b.rle;
			for (uint32_t i = 0; i < nrle; i++) {
				const uint32_t s = rle[2 * i];
				bw.put(S.u.b.code_cl[s], S.u.b.len_cl[s]);
				if (s == 17) {
					bw.put(rle[2 * i + 1], 3);
				} else if (s == 18) {
					bw.put(rle[2 * i + 1], 7);
				}
			}
		}
		uint32_t wpos = __shfl_sync(0xFFFFFFFFu, bw.wpos, 0);
		uint32_t carry = __shfl_sync(0xFFFFFFFFu, (uint32_t)bw.acc, 0);
		uint32_t off0 = __shfl_sync(0xFFFFFFFFu, bw.nacc, 0);
		uint32_t *out32 = reinterpret_cast<uint32_t *>(co);
		for (uint32_t base = 0; base < ntok; base += 32) {
			uint64_t v = 0;
			uint32_t nb = 0;
			if (base + lane < ntok) {
				const uint32_t tk = tok[base + lane];
				if (tk & 0x80000000u) {
					uint32_t xb, xv;
					const uint32_t ls = dfl_len_sym(tk & 0xFFu, xb, xv);
					v = S.u.b.code_ll[ls];
					nb = S.u.b.len_ll[ls];
					v |= (uint64_t)xv << nb;
					nb += xb;
					const uint32_t ds = dfl_dist_sym((tk >> 8) & 0x7FFFu, xb, xv);
					v |= (uint64_t)S.u.b.code_d[ds] << nb;
					nb += S.u.b.len_d[ds];
					v |= (uint64_t)xv << nb;
					nb += xb;
				} else {
					v = S.u.b.code_ll[tk];
					nb = S.u.b.len_ll[tk];
				}
			}
			uint32_t incl = nb;
			for (int o = 1; o < 32; o <<= 1) {
				const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
				if (lane >= o) {
					incl += y;
				}
			}
			const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
			for (int i = lane; i < 72; i += 32) {
				S.u.b.stage[i] = (i == 0) ? carry : 0u;
			}
			__syncwarp();
			if (nb) {
				const uint32_t o = off0 + incl - nb;
				const uint32_t wi = o >> 5, sh = o & 31u;
				atomicOr(&S.u.b.stage[wi], (uint32_t)(v << sh));
				const uint64_t hi = sh ? (v >> (32 - sh)) : (v >> 32);
				if (sh + nb > 32) {
					atomicOr(&S.u.b.stage[wi + 1], (uint32_t)hi);
				}
				if (sh + nb > 64) {
					atomicOr(&S.u.b.stage[wi + 2], (uint32_t)(hi >> 32));
				}
			}
			__syncwarp();
			const uint32_t endbit = off0 + total;
			const uint32_t nfull = endbit >> 5;
			for (uint32_t i = lane; i < nfull; i += 32) {
				out32[wpos + i] = S.u.b.stage[i];
			}
			carry = S.u.b.stage[nfull];
			wpos += nfull;
			off0 = endbit & 31u;
			__syncwarp();
		}
		if (lane == 0) {
			bw.wpos = wpos;
			bw.acc = carry;
			bw.nacc = off0;
			bw.put(S.u.b.code_ll[256], S.u.b.len_ll[256]);   // end of block
			bw.put(ck.last & 1u, 3);              // empty stored block: BFINAL, BTYPE=00
			if (bw.nacc & 7) {
				bw.put(0, 8 - (bw.nacc & 7));           // pad to a byte boundary
			}
			bw.put(0x0000u, 16);
			bw.put(0xFFFFu, 16);
			// flush the remaining whole bytes
			uint32_t nbytes = bw.wpos * 4;
			uint8_t *tail = co + nbytes;
			while (bw.nacc) {
				*tail++ = (uint8_t)bw.acc;
				bw.acc >>= 8;
				bw.nacc -= 8;
				nbytes++;
			}
			S.misc[1] = nbytes;
		}
		__syncwarp();
		out_bytes = S.misc[1];
	}
	if (lane == 0) {
		csize[ci] = out_bytes;
	}
	__syncwarp();
}

// grid: persistent; one warp per chunk, chunks handed out in order.
#define DFL_WARPS 3   // warps per CTA: seven CTAs (21 chunks) fit the shared memory of an SM
// ZSTD: the job holds method-93 entries (their chunks become Zstandard blocks); a pure DEFLATE job runs the instantiation without that path
template <bool ZSTD>
__global__ void __launch_bounds__(32 * DFL_WARPS) k_deflate_chunks(const uint8_t *__restrict__ in, const OtzDflChunk *__restrict__ chunks, uint32_t n_chunks,
	uint32_t *__restrict__ tokens /* DFL_CHUNK per chunk slot */, uint8_t *__restrict__ cout, uint32_t *__restrict__ csize,
	uint32_t *__restrict__ work_counter, uint32_t n_slots) {
	extern __shared__ __align__(16) uint8_t smem_raw[];
	const int lane = threadIdx.x & 31;
	const int warp = threadIdx.x >> 5;
	DeflateSmem &S = reinterpret_cast<DeflateSmem *>(smem_raw)[warp];
	const uint32_t slot = blockIdx.x * (blockDim.x >> 5) + warp;   // token scratch slot of this warp
	uint32_t *tok = tokens + (uint64_t)slot * DFL_CHUNK;
	(void)n_slots;
	for (;;) {
		uint32_t ci = 0;
		if (lane == 0) {
			ci = atomicAdd(work_counter, 1u);
		}
		ci = __shfl_sync(0xFFFFFFFFu, ci, 0);
		if (ci >= n_chunks) {
			break;
		}
		const OtzDflChunk ck = chunks[ci];
		const uint32_t n = ck.len;
		const bool fast = (ck.last & 8u) != 0u;   // compression level 1: first pass only
		const uint64_t ia = reinterpret_cast<uint64_t>(in + ck.in_ofs);
		const uint32_t *w = reinterpret_cast<const uint32_t *>(ia & ~3ull);
		const uint32_t sh0 = (uint32_t)(ia & 3ull);   // byte x of the chunk lives at word-array byte sh0 + x
		uint8_t *co = cout + (uint64_t)ci * DFL_OUT_STRIDE;

		// ---------------- phase 1: LZ77
		for (int i = lane; i < (1 << DFL_HASH_BITS) / 2; i += 32) {
			reinterpret_cast<uint32_t *>(S.u.ht)[i] = 0;
		}
		for (int i = lane; i < 288; i += 32) {
			S.hist_ll[i] = 0;
		}
		S.hist_d[lane] = 0;
		if (lane < 4) {
			S.misc[lane] = 0;
		}
		__syncwarp();
		uint32_t ntok = 0;   // tokens emitted (uniform)
		uint32_t cur = 0;
		while (cur < n) {
			const uint32_t p = cur + lane;
			uint32_t mlen = 0, mdist = 0;
			const bool can = p + DFL_MIN_MATCH <= n;
			uint32_t h = 0, v = 0;
			// default: the hash table is 512 buckets of the last DFL_WAYS earlier positions with this hash (position + 1, 0 = none;
			// most recent in the low half of .x).  Fast entries: 4,096 single slots under a 12-bit hash.
			uint4 bk = make_uint4(0u, 0u, 0u, 0u);
			if (can) {
				v = dfl_word(w, sh0 + p);
				if (fast) {
					h = (v * 2654435761u) >> (32 - DFL_HASH_BITS);
					bk.x = S.u.ht[h];
				} else {
					h = (v * 2654435761u) >> (32 - DFL_BUCKET_BITS);
					bk = *reinterpret_cast<const uint4 *>(&S.u.ht[DFL_WAYS * h]);
				}
			}
			// same-hash lanes: the highest lane (latest position) records itself, deterministically; a bucket moves up by one way
			const uint32_t same = __match_any_sync(0xFFFFFFFFu, can ? h : 0xFFFFFFFFu);
			if (can && lane == 31 - __clz(same)) {
				if (fast) {
					S.u.ht[h] = (uint16_t)(p + 1u);
				} else {
					*reinterpret_cast<uint4 *>(&S.u.ht[DFL_WAYS * h]) =
						make_uint4((bk.x << 16) | (p + 1u), (bk.y << 16) | (bk.x >> 16), (bk.z << 16) | (bk.y >> 16), (bk.w << 16) | (bk.z >> 16));
				}
			}
			// FIRST PASS: the most recent occurrence, for every position (16 bytes per trip: the ten word loads of a trip are in
			// flight together, a trip costs one round trip to L1 / L2; the bytes read beyond maxl lie inside the padded input
			// buffer and are cut off below)
			const uint32_t maxl = can ? min((uint32_t)DFL_MAX_MATCH, n - p) : 0u;
			{
				const uint32_t cand = bk.x & 0xFFFFu;
				if (can && cand && p - (cand - 1u) <= 32768u) {   // RFC 1951 window
					const uint32_t l = dfl_extend(w, sh0, cand - 1u, p, maxl);
					if (l >= DFL_MIN_MATCH) {
						mlen = l;
						mdist = p - (cand - 1u);
					}
				}
			}
			// SECOND PASS (not for fast entries): the other seven ways, but only for the positions where the parse of the first
			// pass starts a token — about a third of them; the rest lies inside a match and is skipped whatever its candidates
			// are.  The (token, way) pairs are dealt to the 32 lanes, so a round of the extension loop works on 32 candidates
			// whatever their owners; a candidate that cannot beat the owner's match is dropped after ONE 4-byte comparison (the
			// bytes that would make it longer: zlib's scan_end test — a 9-bit hash sends many strangers into a bucket).
			if (!fast) {
				const uint32_t lim1 = min(32u, n - cur);
				uint32_t i1 = 0, t1 = 0, spos = 0;
				while (i1 < lim1) {
					const uint32_t L = __shfl_sync(0xFFFFFFFFu, mlen, i1 & 31u);
					const uint32_t Ln = (i1 + 1 < 32) ? __shfl_sync(0xFFFFFFFFu, mlen, (i1 + 1) & 31) : 0u;
					const uint32_t Ln2 = (i1 + 2 < 32) ? __shfl_sync(0xFFFFFFFFu, mlen, (i1 + 2) & 31) : 0u;
					if ((uint32_t)lane == t1) {
						spos = i1;
					}
					t1++;
					i1 += (L >= DFL_MIN_MATCH && Ln <= L && Ln2 <= L + 1u) ? L : 1u;
				}
				S.best[lane] = 0u;
				__syncwarp();
				const uint32_t npairs = (DFL_WAYS - 1) * t1;
				for (uint32_t q0 = 0; q0 < npairs; q0 += 32) {
					const uint32_t q = q0 + lane;
					const bool act = q < npairs;
					const uint32_t tt = act ? q / (DFL_WAYS - 1) : 0u, wy = 1u + q % (DFL_WAYS - 1);
					const uint32_t io = __shfl_sync(0xFFFFFFFFu, spos, tt);   // the owner: window position (= lane) of token tt
					const uint32_t ox = __shfl_sync(0xFFFFFFFFu, bk.x, io), oy = __shfl_sync(0xFFFFFFFFu, bk.y, io);
					const uint32_t oz = __shfl_sync(0xFFFFFFFFu, bk.z, io), ow = __shfl_sync(0xFFFFFFFFu, bk.w, io);
					const uint32_t om = __shfl_sync(0xFFFFFFFFu, mlen, io), ov = __shfl_sync(0xFFFFFFFFu, v, io);
					const uint32_t word = wy < 2 ? ox : wy < 4 ? oy : wy < 6 ? oz : ow;
					const uint32_t cand = (wy & 1u) ? word >> 16 : word & 0xFFFFu;
					const uint32_t po = cur + io;
					const uint32_t omax = po + DFL_MIN_MATCH <= n ? min((uint32_t)DFL_MAX_MATCH, n - po) : 0u;
					bool go = act && cand && po - (cand - 1u) <= 32768u && om < omax;
					const uint32_t c = cand - 1u;
					OTZ_CHK(!go || (io < 32u && c < po && po < n), OTZ_CK_DFL_PAIR);
					if (go) {
						// bytes [t, t + 4) of both strings with t = max(om - 3, 0): equal for every candidate that matches om + 1 bytes
						const uint32_t t = om >= DFL_MIN_MATCH ? om - 3u : 0u;
						go = dfl_word(w, sh0 + c + t) == (t ? dfl_word(w, sh0 + po + t) : ov);
					}
					if (__any_sync(0xFFFFFFFFu, go)) {
						if (go) {
							const uint32_t l = dfl_extend(w, sh0, c, po, omax);
							if (l >= DFL_MIN_MATCH && l > om) {
								atomicMax(&S.best[io], (l << 16) | (32768u - (po - c)));   // (equal lengths: the nearer one)
							}
						}
					}
				}
				__syncwarp();
				const uint32_t bb = S.best[lane];
				if ((bb >> 16) > mlen) {
					mlen = bb >> 16;
					mdist = 32768u - (bb & 0xFFFFu);
				}
			}
			__syncwarp();
			// greedy parse of the 32 positions with two-step lazy evaluation
			uint32_t i = 0, t = 0, mytok = 0;
			const uint32_t lim = min(32u, n - cur);
			while (i < lim) {
				uint32_t L = __shfl_sync(0xFFFFFFFFu, mlen, i);
				const uint32_t Ln = (i + 1 < 32) ? __shfl_sync(0xFFFFFFFFu, mlen, (i + 1) & 31) : 0u;
				const uint32_t Ln2 = (i + 2 < 32) ? __shfl_sync(0xFFFFFFFFu, mlen, (i + 2) & 31) : 0u;
				uint32_t tokv;
				if (L >= DFL_MIN_MATCH && Ln <= L && Ln2 <= L + 1u) {   // (a literal or two are worth a clearly longer match behind them)
					const uint32_t D = __shfl_sync(0xFFFFFFFFu, mdist, i);
					tokv = 0x80000000u | ((D - 1) << 8) | (L - 3);
					i += L;
				} else {
					tokv = 0x40000000u | i;   // literal of window position i; byte fetched below
					i += 1;
				}
				if ((uint32_t)lane == t) {
					mytok = tokv;
				}
				t++;
			}
			// materialise tokens, histogram, coalesced token store
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
					const uint32_t wp = mytok & 31u;
					const uint32_t byte = dfl_word(w, sh0 + cur + wp) & 0xFFu;
					mytok = byte;
					atomicAdd(&S.hist_ll[byte], 1u);
				}
				tok[ntok + lane] = mytok;
			}
			ntok += t;
			cur += i;
		}
		__syncwarp();
		if (ZSTD && (ck.last & 4u)) {
			// method 93: the same tokens as one Zstandard block (k_zstd_enc.cuh)
			const uint32_t ob = zse_emit_block(in + ck.in_ofs, n, tok, ntok, co, (ck.last & 2u) != 0u, (ck.last & 1u) != 0u, ck.pad, lane);
			if (lane == 0) {
				csize[ci] = ob;
			}
			__syncwarp();
			continue;
		}
		dfl_code_emit(S, tok, ntok, in, ck, co, csize, ci);
	}
}

// ---- per-entry totals, STORE fallback decision (otezip.c:793-801, :846-850) and chunk destinations.
struct OtzDflEntry {
	uint64_t in_ofs;
	uint32_t len;
	uint32_t first_chunk;
	uint32_t n_chunks;
	uint16_t method_in;
	uint16_t pad;
};

__global__ void k_deflate_entry_sizes(const OtzDflEntry *__restrict__ ents, uint32_t n, const uint32_t *__restrict__ csize,
	uint32_t *__restrict__ out_size, uint16_t *__restrict__ method_out) {
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) {
		return;
	}
	const OtzDflEntry e = ents[i];
	uint64_t tot = 0;
	const bool coded = e.method_in == OTZ_M_DEFLATE || e.method_in == OTZ_M_ZSTD;
	if (coded) {
		for (uint32_t k = 0; k < e.n_chunks; k++) {
			tot += csize[e.first_chunk + k];
		}
	}
	const bool smaller = coded && e.len > 0 && tot < e.len;   // otezip.c:846-850 / :894-899: a stream that is not smaller is stored
	method_out[i] = smaller ? e.method_in : OTZ_M_STORE;
	out_size[i] = smaller ? (uint32_t)tot : e.len;
}

// exclusive scan of out_size[] into out_ofs[] (single CTA; n <= a few hundred thousand)
__global__ void __launch_bounds__(1024) k_deflate_scan(const uint32_t *__restrict__ out_size, uint32_t n, uint64_t *__restrict__ out_ofs,
	uint64_t *__restrict__ total) {
	__shared__ uint64_t part[1024];
	const uint32_t per = (n + 1023) / 1024;
	const uint32_t b = threadIdx.x * per, e = min(n, b + per);
	uint64_t s = 0;
	for (uint32_t i = b; i < e; i++) {
		s += out_size[i];
	}
	part[threadIdx.x] = s;
	__syncthreads();
	if (threadIdx.x == 0) {
		uint64_t acc = 0;
		for (int i = 0; i < 1024; i++) {
			const uint64_t t = part[i];
			part[i] = acc;
			acc += t;
		}
		*total = acc;
	}
	__syncthreads();
	uint64_t acc = part[threadIdx.x];
	for (uint32_t i = b; i < e; i++) {
		out_ofs[i] = acc;
		acc += out_size[i];
	}
}

// gather: one warp per chunk copies either the compressed slot or the raw bytes to the dense arena
__global__ void __launch_bounds__(256) k_deflate_gather(const uint8_t *__restrict__ in, const uint8_t *__restrict__ cout,
	const OtzDflChunk *__restrict__ chunks, uint32_t n_chunks, const OtzDflEntry *__restrict__ ents, const uint32_t *__restrict__ csize,
	const uint16_t *__restrict__ method_out, const uint64_t *__restrict__ out_ofs, uint8_t *__restrict__ dense) {
	const uint32_t warps_per_cta = blockDim.x >> 5;
	const uint32_t total_warps = gridDim.x * warps_per_cta;
	const int lane = threadIdx.x & 31;
	for (uint32_t c = blockIdx.x * warps_per_cta + (threadIdx.x >> 5); c < n_chunks; c += total_warps) {
		const OtzDflChunk ck = chunks[c];
		const OtzDflEntry e = ents[ck.entry];
		const uint32_t k = c - e.first_chunk;
		if (method_out[ck.entry] != OTZ_M_STORE) {
			uint64_t off = 0;
			for (uint32_t j = lane; j < k; j += 32) {
				off += csize[e.first_chunk + j];
			}
			for (int o = 16; o > 0; o >>= 1) {
				off += __shfl_xor_sync(0xFFFFFFFFu, off, o);
			}
			tile_copy<32>(dense + out_ofs[ck.entry] + off, cout + (uint64_t)c * DFL_OUT_STRIDE, csize[c], lane);
		} else {
			tile_copy<32>(dense + out_ofs[ck.entry] + (uint64_t)k * DFL_CHUNK, in + ck.in_ofs, ck.len, lane);
		}
	}
}

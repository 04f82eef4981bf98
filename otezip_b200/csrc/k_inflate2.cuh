// k_inflate2.cuh — phase B of the two-phase batched raw-DEFLATE (RFC 1951) decoder: the LZ77 executor, plus what the
// two phases share (table format and builder, token format, segment tables of huge streams).
//
// Replaces the copy half of inflate() as driven by otezip_extract_entry
// (/root/reference/src/lib/otezip.c:503-529; decoder src/lib/deflate-dec.inc.c:547-831, "dec" below; the byte-wise
// window copy is dec:521-545).  The decoder is split the way the work parallelises:
//
//   phase A  k_inflate_spec (k_inflate3.cuh)   entropy decoding: one warp (or, for huge streams, one 4-warp CTA) per
//            stream, 32 / 128 pieces of the stream decoded speculatively in parallel, synchronised on symbol boundaries;
//            emits, per stream, the literal bytes (dense) and one 32-bit sequence record per match
//            {literal run : 9, length-3 : 8, distance-1 : 15}.  The 16-bit two-level tables (9-bit / 7-bit roots) are built
//            by the warp from the code lengths (i2_build_table below: canonical order by match_any ranks, every table slot
//            computed independently from the 15-bit left-aligned code boundaries).
//   phase B  k_inflate_lz    one warp per stream executes the sequences: 32 records per coalesced load, warp
//            prefix sums give every record its literal and output position; two batches are in flight — while
//            batch k executes, batch k+1 has been scanned, the descriptor of every match sits in its lane's registers
//            and the sources of its far matches (those that left the shared-memory ring) are on their way into a
//            staging buffer behind the ring by cp.async — so executing a batch touches shared memory only; the
//            matches run in stream order, three shuffles and up to 64 elements per step; completed 512-byte
//            segments leave as coalesced 16-byte stores.  The same kernel executes Zstandard sequences (8-byte
//            records, k_zstd.cuh) and the segments of huge streams over 16-bit symbols (below).
//
// Phase A only commits streams that are plainly valid: final block reached, exactly uncomp_size bytes, regular
// stored-block headers (their payload joins the literals), tables within the fixed budget.  Anything else (errors,
// short streams, exotic code sets) is appended to a fallback list and decoded from scratch by k_inflate, whose
// status words define the behaviour in those cases; the two kernels agree bit for bit on every stream both
// can decode, so the split is invisible to the caller.  The reference's end-of-input rule (dec:811-816,
// SURVEY.md F1) is evaluated in phase A and reported as OTZ_STF_REF_EOB exactly as k_inflate reports it.
#pragma once
#include "otz_common.cuh"
#include "k_inflate.cuh"
#include <type_traits>

#ifndef OTZ_BYTE_STAGE_VECS
#define OTZ_BYTE_STAGE_VECS 64u
#endif
#ifndef OTZ_PAR_STAGE_VECS
#define OTZ_PAR_STAGE_VECS 96u
#endif
#define I2_LIT_ROOT 9
#define I2_DST_ROOT 7
#define I2_LIT_CAP 704   // 512 root slots + 192 second-level slots
#define I2_DST_CAP 192   // 128 root slots + 64 second-level slots

// 16-bit entries.  tb = bits the symbol consumes at this table level INCLUDING its extra bits, so the bit
// position advances by one field of the entry; what the extra bits mean is worked out off the critical path.
//   literal/length table: [3:0] tb, [5:4] kind, then  LIT: [13:6] byte   LEN: [8:6] extra bits, [13:9] symbol-257
//                         LINK: tb = 0, [8:6] index bits of the second-level table (0 = invalid code),
//                               [15:9] (its offset - 512) / 2   (second-level tables are even-sized and packed)
//   distance table:       [4:0] tb, [8:5] extra bits, [13:9] symbol, [15:14] kind (0 = symbol, 3 = LINK/invalid)
//                         LINK: tb = 0, [8:5] index bits (0 = invalid code), [13:9] (offset - 128) / 2
// A LINK entry has tb = 0: the straight-line decoder may add every entry's tb to the bit position blindly.
#define I2_K_LIT 0u
#define I2_K_LEN 1u
#define I2_K_EOB 2u
#define I2_K_LINK 3u
#define I2_LIT_ENTRY(tb, kind, rest) ((uint16_t)((tb) | ((kind) << 4) | ((rest) << 6)))
#define I2_LIT_LINK(bits, off) I2_LIT_ENTRY(0u, I2_K_LINK, (bits) | ((((off) - (1u << I2_LIT_ROOT)) >> 1) << 3))
#define I2_LIT_INVALID I2_LIT_ENTRY(0u, I2_K_LINK, 0u)
#define I2_LIT_LINK_BITS(e) (((e) >> 6) & 7u)
#define I2_LIT_LINK_OFS(e) ((1u << I2_LIT_ROOT) + (((e) >> 9) << 1))
#define I2_DST_ENTRY(tb, xb, sym) ((uint16_t)((tb) | ((xb) << 5) | ((sym) << 9)))
#define I2_DST_LINK(bits, off) ((uint16_t)(((bits) << 5) | ((((off) - (1u << I2_DST_ROOT)) >> 1) << 9) | (3u << 14)))
#define I2_DST_INVALID I2_DST_LINK(0u, (1u << I2_DST_ROOT))
#define I2_DST_LINK_BITS(d) (((d) >> 5) & 15u)
#define I2_DST_LINK_OFS(d) ((1u << I2_DST_ROOT) + ((((d) >> 9) & 31u) << 1))

// sequence record: [8:0] literal run, [16:9] match length - 3, [31:17] distance - 1
#define I2_SEQ_ESC 511u   // literal run of exactly 511 bytes and no match

struct I2TokRes {
	uint32_t nseq;    // sequence records written (descending from the end of the stream's scratch)
	uint32_t nlit;    // literal bytes written (ascending from the start)
	int32_t status;   // status word to report when phase B has produced the bytes
	uint32_t ok;      // 1: phase B executes this stream; 0: it went to the fallback list
};


// worst-case scratch of a stream of n output bytes: literals + 4 bytes per match (>= 3 bytes each) + escapes
__host__ __device__ __forceinline__ uint64_t i2_scratch_bytes(uint64_t n) {
	return ((n + 4 * (n / 3 + n / 511 + 4) + 16 + 15) / 16) * 16;
}

// length / distance bases (dec:720-725, dec:766-771) from the symbol
__device__ __forceinline__ uint32_t i2_len_base(uint32_t v, uint32_t xb) {
	return v < 8u ? 3u + v : v == 28u ? 258u : 3u + ((4u + (v & 3u)) << xb);
}
__device__ __forceinline__ uint32_t i2_dist_base(uint32_t ds, uint32_t xb) { return ds < 4u ? 1u + ds : 1u + ((2u + (ds & 1u)) << xb); }

// ------------------------------------------------------------------------------------------------
// Warp-cooperative build of one two-level table from code lengths held in registers.
// lens[j] = code length of combined symbol 32*j + lane (literal/length alphabet first, then distances);
// this call covers combined symbols [b0, b0 + n).  Returns 0 ok, 1 = not usable on the fast path
// (invalid / incomplete set in a shape k_inflate has to judge, or second-level budget exceeded).
template <bool IS_DIST>
__device__ __forceinline__ uint16_t i2_symbol_entry(uint32_t s, uint32_t cb) {
	if (IS_DIST) {
		const uint32_t xb = s < 4u ? 0u : (s - 2u) >> 1;
		return s < 30u ? I2_DST_ENTRY(cb + xb, xb, s) : I2_DST_INVALID;
	}
	if (s < 256u) {
		return I2_LIT_ENTRY(cb, I2_K_LIT, s);
	}
	if (s == 256u) {
		return I2_LIT_ENTRY(cb, I2_K_EOB, 0u);
	}
	const uint32_t v = s - 257u;
	const uint32_t xb = (v < 8u || v == 28u) ? 0u : (v - 4u) >> 2;
	return s < 286u ? I2_LIT_ENTRY(cb + xb, I2_K_LEN, xb | (v << 3)) : I2_LIT_INVALID;
}

// length and position in sorted[] of the code that covers the 15-bit left-aligned value c15 (len 16 = none);
// lim[j] = S.limit15[j], held in registers by the caller
template <typename WS>
__device__ __forceinline__ void i2_lookup15(const WS &S, const uint32_t (&lim)[16], uint32_t c15, uint32_t &len, uint32_t &idx) {
	uint32_t l = 1;
#pragma unroll
	for (int j = 1; j <= 15; j++) {
		l += (c15 >= lim[j]);
	}
	len = l;
	const uint32_t ll = l > 15u ? 15u : l;
	idx = S.offs[ll] + ((c15 - S.first15[ll]) >> (15u - ll));
}

template <bool IS_DIST, int ROOT, int CAP, typename WS>
__device__ __noinline__ int i2_build_table(WS &S, const uint32_t (&lens)[10], uint32_t b0, uint32_t n, uint16_t *tbl) {
	const uint32_t lane = threadIdx.x & 31u;
	constexpr uint16_t INVALID = IS_DIST ? I2_DST_INVALID : I2_LIT_INVALID;
	if (lane < 16) {
		S.cnt[lane] = 0;
	}
	__syncwarp();
	uint32_t mylen[10];
#pragma unroll
	for (int j = 0; j < 10; j++) {
		const uint32_t s = 32u * j + lane - b0;
		mylen[j] = s < n ? lens[j] : 0u;
		if (mylen[j]) {
			atomicAdd(&S.cnt[mylen[j]], 1u);
		}
	}
	__syncwarp();
	int left = 1;
	uint32_t ncodes = 0;
	{
		uint32_t code = 0, off = 0;
		for (uint32_t l = 1; l <= 15; l++) {
			const uint32_t c = S.cnt[l];
			left = (left << 1) - (int)c;
			if (left < 0) {
				return 1;   // over-subscribed
			}
			code = (code + (l > 1 ? S.cnt[l - 1] : 0u)) << 1;
			if (lane == 0) {
				S.offs[l] = off;
				S.run[l] = off;
				S.first15[l] = code << (15u - l);
				S.limit15[l] = (code + c) << (15u - l);
			}
			off += c;
			ncodes += c;
		}
	}
	constexpr uint32_t ROOTSZ = 1u << ROOT;
	if (ncodes == 0) {
		if (!IS_DIST) {
			return 1;
		}
		for (uint32_t k = lane; k < ROOTSZ; k += 32) {
			tbl[k] = INVALID;   // a block of literals only: any distance code is an error
		}
		__syncwarp();
		return 0;
	}
	if (left > 0 && !(ncodes == 1 && S.cnt[1] == 1)) {
		return 1;   // incomplete set (zlib accepts only a single 1-bit code): k_inflate reports it
	}
	__syncwarp();
	// canonical order: sorted[] = symbols by (length, symbol)
#pragma unroll
	for (int j = 0; j < 10; j++) {
		const uint32_t l = mylen[j];
		const uint32_t m = __match_any_sync(0xFFFFFFFFu, l);
		const uint32_t rank = __popc(m & ((1u << lane) - 1u));
		if (l) {
			S.sorted[S.run[l] + rank] = (uint16_t)(32u * j + lane - b0);
		}
		__syncwarp();
		if (l && rank == 0) {
			S.run[l] += __popc(m);
		}
		__syncwarp();
	}
	// root slots: slot k holds the code whose bits, LSB first, are a prefix of k
	uint32_t lim[16];
#pragma unroll
	for (int j = 0; j < 16; j++) {
		lim[j] = S.limit15[j];
	}
	const uint32_t long15 = S.limit15[ROOT];          // first 15-bit value whose code is longer than ROOT bits
	const uint32_t end15 = S.limit15[15];             // one past the last covered value (32768 when complete)
	for (uint32_t k = lane; k < ROOTSZ; k += 32) {
		const uint32_t c15 = (__brev(k) >> (32 - ROOT)) << (15 - ROOT);
		uint16_t e = INVALID;
		if (c15 < long15) {
			uint32_t len, idx;
			i2_lookup15(S, lim, c15, len, idx);
			e = i2_symbol_entry<IS_DIST>(S.sorted[idx], len);
		}
		tbl[k] = e;
	}
	// prefixes of codes longer than ROOT bits: one second-level table each, sized by its longest code
	if (end15 > long15) {
		const uint32_t p0 = long15 >> (15 - ROOT), p1 = (end15 + (1u << (15 - ROOT)) - 1u) >> (15 - ROOT);
		uint32_t next_free = ROOTSZ;
		for (uint32_t pb = p0; pb < p1; pb += 32) {
			const uint32_t p = pb + lane;
			uint32_t sub_bits = 0;
			if (p < p1) {
				uint32_t v15 = ((p + 1u) << (15 - ROOT)) - 1u;
				v15 = v15 < end15 ? v15 : end15 - 1u;
				uint32_t len, idx;
				i2_lookup15(S, lim, v15, len, idx);
				sub_bits = len - ROOT;
			}
			const uint32_t size = p < p1 ? (1u << sub_bits) : 0u;
			uint32_t incl = size;
#pragma unroll
			for (int d = 1; d < 32; d <<= 1) {
				const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
				if ((int)lane >= d) {
					incl += t;
				}
			}
			const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
			if (next_free + total > (uint32_t)CAP) {
				return 1;   // second-level budget exceeded: k_inflate (worst-case tables) takes the stream
			}
			const uint32_t sub_off = next_free + incl - size;
			next_free += total;
			if (p < p1) {
				tbl[__brev(p) >> (32 - ROOT)] = IS_DIST ? I2_DST_LINK(sub_bits, sub_off) : I2_LIT_LINK(sub_bits, sub_off);
				for (uint32_t t = 0; t < size; t++) {
					const uint32_t c15 = (p << (15 - ROOT)) | ((__brev(t) >> (32u - sub_bits)) << (15u - ROOT - sub_bits));
					uint16_t e = INVALID;
					if (c15 < end15) {
						uint32_t len, idx;
						i2_lookup15(S, lim, c15, len, idx);
						e = i2_symbol_entry<IS_DIST>(S.sorted[idx], len - ROOT);
					}
					tbl[sub_off + t] = e;
				}
			}
		}
	}
	__syncwarp();
	return 0;
}

// ------------------------------------------------------------------------------------------------
// HUGE streams.  One warp executing the sequences of a 16 MiB entry one after the other would set the critical path
// of a whole batch (~100 ms), so phase A cuts the token stream of a huge entry into SEGMENTS (at round boundaries,
// each behind a match, >= 256 KiB of output; it knows every output position) and fills the tables below; k_seg_stitch
// checks the chain once more (the sizes add up, no match reaches before the stream) and places the segments in the
// symbol buffer; k_inflate_lz<.., PAR> executes every segment on its own warp over 16-bit symbols.  A chain that does
// not close sends the stream to k_inflate like every other declined stream.
#define I2_MAXSEG 256
#define I2_PREWIN 32768u   // elements of history a segment may refer to (DEFLATE window)
#define I2_SEGF_OK 1u
#define I2_SEGF_FINAL 2u
#define I2_SEGF_DEAD 4u
#define I2_SEGF_REF_EOB 8u

struct I2SegRes {
	uint32_t nseq, nlit;    // tokens of the segment
	uint32_t produced;      // output bytes of the segment
	uint32_t end_bit;       // bit position (in the stream) where the segment stopped
	uint32_t reach;         // how far a match reaches before the segment's first output byte
	uint32_t flags;         // I2_SEGF_*
	uint64_t scr_lo, scr_hi;   // its slice of the stream's token scratch (literals up from lo, records down from hi)
};

struct I2SegCtl {
	uint32_t *count;     // [n_huge] segments of the stream
	uint32_t *start;     // [n_huge][I2_MAXSEG] start mark of every segment, ascending, [0] = 0 (= end mark of the one before)
	I2SegRes *res;       // [n_huge][I2_MAXSEG]
	uint32_t *live;      // [n_huge][I2_MAXSEG] the chain of segments that make up the stream
	uint32_t *nlive;     // [n_huge] length of the chain (0 = the stream was declined)
	int32_t *seg_status; // [n_huge] status word of an accepted stream
	// parallel execution of the chain (k_inflate_lz<.., PAR> + k_seg_window + k_seg_translate)
	uint32_t *par;       // [n_huge] 1 = the segments of the stream are executed in parallel into the symbol buffer
	uint32_t *par_items; // work list: stream << 16 | position in the chain
	uint32_t *n_par;
	uint64_t *sym_start; // [n_huge][I2_MAXSEG] by chain position: first element of the segment in the symbol buffer
	uint32_t *out_start; // [n_huge][I2_MAXSEG] by chain position: first output byte of the segment in the entry
	unsigned long long *sym_top;   // bump allocator of the symbol buffer (elements)
	uint64_t sym_cap;    // its capacity (0 = no parallel execution)
	uint32_t out_mis;    // address of the output arena & 15
};

// One thread per huge stream: follow the chain of segments.  The stream is accepted (nlive > 0) only if every link
// fits; otherwise it is appended to the fallback list of k_inflate.
//
// An accepted stream with more than one segment gets room in the symbol buffer (if there is any left): per segment
// I2_PREWIN marker elements, then its output as 16-bit symbols, placed so that symbol i of the segment and output byte i
// have the same index modulo 16 (k_seg_translate works on whole vectors of both).
__global__ void k_seg_stitch(const otz_entry *__restrict__ ents, const int32_t *__restrict__ status, const uint32_t *__restrict__ list,
	uint32_t n_huge, I2SegCtl seg, uint32_t *__restrict__ fb_list, uint32_t *__restrict__ fb_count, uint32_t h0) {
	const uint32_t h = h0 + blockIdx.x * blockDim.x + threadIdx.x;   // streams [h0, n_huge) of the list: one group of huge streams
	if (h >= n_huge) {
		return;
	}
	const uint32_t ei = list[h];
	if (OTZ_ST_CODE(status[ei]) != OTZ_ST_OK) {
		return;
	}
	const uint32_t n = seg.count[h], cap = ents[ei].uncomp_size;
	const I2SegRes *res = seg.res + h * I2_MAXSEG;
	const uint32_t *st = seg.start + h * I2_MAXSEG;
	uint32_t *live = seg.live + h * I2_MAXSEG;
	uint32_t j = 0, nlive = 0;
	uint64_t out = 0;
	bool ok = true, done = false, ref_eob = false;
	while (ok && !done) {
		const I2SegRes r = res[j];
		if (!(r.flags & I2_SEGF_OK) || r.reach > out || out + r.produced > cap) {
			ok = false;
			break;
		}
		live[nlive++] = j;
		out += r.produced;
		if (r.flags & I2_SEGF_FINAL) {
			done = true;
			ref_eob = (r.flags & I2_SEGF_REF_EOB) != 0u;
			break;
		}
		uint32_t jn = j + 1;
		while (jn < n && st[jn] < r.end_bit) {
			jn++;
		}
		if (jn >= n || st[jn] != r.end_bit) {
			ok = false;
			break;
		}
		j = jn;
	}
	if (ok && done && out == cap) {
		seg.nlive[h] = nlive;
		seg.seg_status[h] = OTZ_ST_OK | (ref_eob ? OTZ_STF_REF_EOB : 0);
		uint32_t par = 0;
		if (nlive > 1 && seg.sym_cap) {
			const uint64_t need = (uint64_t)cap + (uint64_t)nlive * (I2_PREWIN + 16u);
			const uint64_t base = atomicAdd(seg.sym_top, (unsigned long long)need);
			if (base + need <= seg.sym_cap) {
				par = 1;
				uint64_t at = base;
				uint32_t o = 0;
				const uint32_t omis = (uint32_t)((seg.out_mis + ents[ei].out_ofs) & 15u);
				for (uint32_t c = 0; c < nlive; c++) {
					uint64_t first = at + I2_PREWIN;
					first += ((omis + o) - (uint32_t)first) & 15u;
					seg.sym_start[h * I2_MAXSEG + c] = first;
					seg.out_start[h * I2_MAXSEG + c] = o;
					const uint32_t pr = res[live[c]].produced;
					at += I2_PREWIN + 16u + pr;
					o += pr;
				}
				const uint32_t w = atomicAdd(seg.n_par, nlive);
				for (uint32_t c = 0; c < nlive; c++) {
					seg.par_items[w + c] = (h << 16) | c;
				}
			}
		}
		seg.par[h] = par;
	} else {
		seg.par[h] = 0;
		seg.nlive[h] = 0;
		fb_list[atomicAdd(fb_count, 1u)] = ei;
	}
}

// Parallel execution of a huge stream.  Every segment of the chain is executed by its own warp over 16-bit symbols:
// values below 256 are bytes, 256 + j stands for "byte j of the 32 KiB before this segment", unknown while the
// segments before it are still being executed (k_inflate_lz<.., PAR> prefills those markers and copies them around
// like any other element).  k_seg_window then walks the chain of ONE stream per CTA and resolves only the last
// 32 KiB of every segment — the window of the next one — straight into the output; step c reads what steps < c
// wrote.  k_seg_translate finally resolves everything in front of those tails, all segments at once.
__global__ void __launch_bounds__(1024) k_seg_window(uint8_t *__restrict__ out, const otz_entry *__restrict__ ents, const uint32_t *__restrict__ list,
	uint32_t n_huge, const uint16_t *__restrict__ sym, int32_t *__restrict__ status, uint32_t *__restrict__ produced_out, I2SegCtl seg, uint32_t h0) {
	const uint32_t h = h0 + blockIdx.x;
	if (h >= n_huge || !seg.par[h]) {
		return;
	}
	const uint32_t ei = list[h];
	uint8_t *const o = out + ents[ei].out_ofs;
	const uint32_t nlive = seg.nlive[h];
	for (uint32_t c = 0; c < nlive; c++) {
		const uint32_t pr = seg.res[h * I2_MAXSEG + seg.live[h * I2_MAXSEG + c]].produced;
		const uint32_t os = seg.out_start[h * I2_MAXSEG + c];
		const uint16_t *sp = sym + seg.sym_start[h * I2_MAXSEG + c];
		const uint32_t t0 = pr > I2_PREWIN ? pr - I2_PREWIN : 0u;
		// (two dependent HBM round trips per element — the symbol, then the byte its marker names: eight elements per thread
		// are in flight together)
		for (uint32_t i0 = t0 + threadIdx.x; i0 < pr; i0 += 8u * blockDim.x) {
			uint32_t v[8];
#pragma unroll
			for (int u = 0; u < 8; u++) {
				const uint32_t i = i0 + u * blockDim.x;
				v[u] = i < pr ? __ldcs(sp + i) : 0u;
			}
#pragma unroll
			for (int u = 0; u < 8; u++) {
				// (a marker only exists where a match reached, and k_seg_stitch checked reach <= os)
				v[u] = v[u] < 256u ? v[u] : (uint32_t)__ldcg(o + (os - I2_PREWIN + (v[u] - 256u)));
			}
#pragma unroll
			for (int u = 0; u < 8; u++) {
				const uint32_t i = i0 + u * blockDim.x;
				if (i < pr) {
					o[os + i] = (uint8_t)v[u];
				}
			}
		}
		__syncthreads();
	}
	if (threadIdx.x == 0) {
		status[ei] = seg.seg_status[h];
		produced_out[ei] = ents[ei].uncomp_size;
	}
}

// One CTA per work item (segment): symbols [0, produced - 32 KiB) -> bytes.  The 32 KiB before the segment (final
// since k_seg_window) are staged in shared memory: in text most vectors still hold a marker or two.
#define I2_TR_THREADS 512
// The window — up to 32 KiB + 16 contiguous, 16-byte aligned bytes — is staged by ONE bulk-copy instruction (TMA:
// cp.async.bulk global -> shared, completion counted in bytes on an mbarrier) issued by one thread, instead of 2,049
// vector loads and stores through registers; the other 511 threads go straight to the wait.
__global__ void __launch_bounds__(I2_TR_THREADS) k_seg_translate(uint8_t *__restrict__ out, const otz_entry *__restrict__ ents, const uint32_t *__restrict__ list,
	const uint16_t *__restrict__ sym, uint32_t *__restrict__ work_counter, I2SegCtl seg) {
	__shared__ __align__(16) uint8_t s_win[I2_PREWIN + 16];
	__shared__ __align__(8) uint64_t s_mbar;
	__shared__ uint32_t s_k;
	const uint32_t n = *seg.n_par;
	const uint32_t mbar_sa = (uint32_t)__cvta_generic_to_shared(&s_mbar), win_sa = (uint32_t)__cvta_generic_to_shared(s_win);
	if (threadIdx.x == 0) {
		asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar_sa) : "memory");
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	uint32_t phase = 0;
	for (;;) {
		__syncthreads();
		if (threadIdx.x == 0) {
			s_k = atomicAdd(work_counter, 1u);
		}
		__syncthreads();
		const uint32_t k = s_k;
		if (k >= n) {
			break;
		}
		const uint32_t it = seg.par_items[k], h = it >> 16, c = it & 0xFFFFu;
		const I2SegRes *r_ = &seg.res[h * I2_MAXSEG + seg.live[h * I2_MAXSEG + c]];
		const uint32_t pr = r_->produced;
		if (pr <= I2_PREWIN) {
			continue;
		}
		const uint32_t body = pr - I2_PREWIN, os = seg.out_start[h * I2_MAXSEG + c];
		uint8_t *const o = out + ents[list[h]].out_ofs + os;        // o[i] <- sp[i]
		const uint16_t *const sp = sym + seg.sym_start[h * I2_MAXSEG + c];
		const uint32_t omis = (uint32_t)(reinterpret_cast<uint64_t>(o) & 15u);
		if (r_->reach) {   // (no reach, no markers; and the first segment of a stream has nothing in front of it)
			// (a segment in the first 32 KiB of its entry: nothing is read in front of the entry's output)
			const int64_t avail = (int64_t)os + (int64_t)((reinterpret_cast<uint64_t>(o) - os) & 15u);
			const int64_t lack = (int64_t)(I2_PREWIN + omis) - avail;
			const uint32_t x0 = lack > 0 ? (uint32_t)((lack + 15) >> 4) : 0u;   // first 16-byte vector of the window that exists
			const uint32_t bytes = (I2_PREWIN / 16u + 1u - x0) * 16u;
			if (threadIdx.x == 0) {
				// (the reads of the previous item's window — generic proxy — are ordered before this write by the async proxy)
				asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
				asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar_sa), "r"(bytes) : "memory");
				asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(win_sa + 16u * x0),
					"l"(o - I2_PREWIN - omis + 16u * x0), "r"(bytes), "r"(mbar_sa)
					: "memory");
			}
			uint32_t done = 0;
			do {
				asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
					: "=r"(done)
					: "r"(mbar_sa), "r"(phase)
					: "memory");
			} while (!done);
			phase ^= 1u;
		}
		const uint8_t *const win = s_win + omis;                    // marker j -> win[j]
		const uint32_t head = min(body, (16u - omis) & 15u);
		const uint32_t nvec = (body - head) >> 4, tail0 = head + (nvec << 4);
		for (uint32_t i = threadIdx.x; i < head; i += blockDim.x) {
			const uint32_t v = sp[i];
			o[i] = v < 256u ? (uint8_t)v : win[(v - 256u) & (I2_PREWIN - 1u)];
		}
		for (uint32_t i = tail0 + threadIdx.x; i < body; i += blockDim.x) {
			const uint32_t v = sp[i];
			o[i] = v < 256u ? (uint8_t)v : win[(v - 256u) & (I2_PREWIN - 1u)];
		}
#pragma unroll 2
		for (uint32_t x = threadIdx.x; x < nvec; x += blockDim.x) {
			const uint32_t i = head + (x << 4);
			const uint4 a = __ldcs(reinterpret_cast<const uint4 *>(sp + i)), b = __ldcs(reinterpret_cast<const uint4 *>(sp + i + 8));
			uint32_t w[8] = { a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w };
			uint32_t r[4];
			if (((a.x | a.y | a.z | a.w | b.x | b.y | b.z | b.w) & 0xFF00FF00u) == 0u) {
#pragma unroll
				for (int j = 0; j < 4; j++) {
					r[j] = __byte_perm(w[2 * j], w[2 * j + 1], 0x6420);
				}
			} else {
#pragma unroll
				for (int j = 0; j < 4; j++) {
					uint32_t acc = 0;
#pragma unroll
					for (int t = 0; t < 4; t++) {
						const uint32_t v = (w[2 * j + (t >> 1)] >> (16 * (t & 1))) & 0xFFFFu;
						const uint32_t byte = v < 256u ? v : (uint32_t)win[(v - 256u) & (I2_PREWIN - 1u)];
						acc |= byte << (8 * t);
					}
					r[j] = acc;
				}
			}
			__stcs(reinterpret_cast<uint4 *>(o + i), make_uint4(r[0], r[1], r[2], r[3]));
		}
	}
}

// ------------------------------------------------------------------------------------------------
// phase B.  One warp per committed stream; W = bytes of shared-memory ring per warp.  Ring index of output
// byte p is (p + mis) & (W-1) with mis = dst & 15 (as OutRing in k_inflate.cuh), so ring vectors line up with
// 16-byte aligned global vectors.
//
// The sequence records are executed in batches of up to 32 (one per lane), software-pipelined over two batches:
// while batch k runs, batch k+1 has already been scanned (warp prefix sums give every record its literal and
// output positions), its match descriptors sit in shared memory, the first literals of every run are in
// registers and — the point of the exercise — the sources of its FAR matches (those that left the ring; they
// were flushed to HBM before batch k started, see SPAN_MAX) are on their way into a staging buffer as 16-byte
// cp.async copies.  Executing a batch therefore touches shared memory only.
// The executor is written over an element type T: bytes for ordinary streams, 16-bit SYMBOLS for the segments of a
// huge stream that are executed in parallel (k_seg_window below): positions, distances and lengths are in elements,
// VEC = elements per 16-byte vector.
template <typename T>
struct I2Elem {
	static constexpr uint32_t VEC = 16u / sizeof(T);
	static constexpr uint32_t STAGE_VECS = sizeof(T) == 1 ? OTZ_BYTE_STAGE_VECS : OTZ_PAR_STAGE_VECS;   // staging vectors per batch; a batch ends where they are used up
	static constexpr uint32_t STAGE = STAGE_VECS * VEC;
};

template <bool PAR>
struct I2ElemOf {
	typedef uint8_t type;
};
template <>
struct I2ElemOf<true> {
	typedef uint16_t type;
};

template <int W>
struct I2Ring {
	static constexpr uint32_t MASK = W - 1;
	static constexpr uint32_t SEG = 512;
	// output bytes per batch.  W >= 2 * SPAN_MAX + SEG + 258 guarantees that a far source of batch k+1 has been
	// flushed to HBM before batch k starts (when its copy is issued).
	static constexpr uint32_t SPAN_MAX = W >= 8192 ? 2048u : 1024u;   // (>= 769: a batch always takes at least one record)
	static_assert(W >= 4096, "the ring must hold two batches, a flush segment and one match (see above)");
};

template <int W, typename T = uint8_t>
struct __align__(16) I2LzSmem {
	T ring[W];
	T stage[2][I2Elem<T>::STAGE];   // (directly behind the ring: a match source is ONE index from the ring's base, see I2Batch::mb)
};

// write ring[a, b) (linear positions) to HBM; whole warp, ring contents visible (caller synced)
template <int W, typename T>
__device__ __forceinline__ void i2_flush_range(T *gbase, const T *ring, uint32_t a, uint32_t b, uint32_t lane) {
	constexpr uint32_t MASK = W - 1, VEC = I2Elem<T>::VEC;
	const uint32_t a16 = (a + VEC - 1u) & ~(VEC - 1u), b16 = b & ~(VEC - 1u);
	if (a16 >= b16) {
		for (uint32_t x = a + lane; x < b; x += 32) {
			gbase[x] = ring[x & MASK];
		}
		return;
	}
	for (uint32_t x = a + lane; x < a16; x += 32) {
		gbase[x] = ring[x & MASK];
	}
#pragma unroll 1
	for (uint32_t x = a16 + VEC * lane; x < b16; x += 32u * VEC) {
		*reinterpret_cast<uint4 *>(gbase + x) = *reinterpret_cast<const uint4 *>(ring + (x & MASK));
	}
	for (uint32_t x = b16 + lane; x < b; x += 32) {
		gbase[x] = ring[x & MASK];
	}
}

// overlapping LZ77 copy (distance < length): periodic extension of the last `dd` bytes, whole warp (dec:521-533)
template <int W, typename T>
__device__ __forceinline__ void i2_copy_periodic(T *rb, uint32_t dq, uint32_t sq, uint32_t dd, uint32_t len, uint32_t lane) {
	constexpr uint32_t MASK = W - 1;
	uint32_t r = dd > lane ? lane : lane % dd;
	const uint32_t step = dd > 32u ? 32u : 32u % dd;
	for (uint32_t x = lane; x < len; x += 32) {
		rb[(dq + x) & MASK] = rb[(sq + r) & MASK];
		r += step;
		r = r >= dd ? r - dd : r;
	}
}

__device__ __forceinline__ uint32_t i2_ld_le16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

// one element at shared-memory byte address sa + OFS, loaded into / stored from a 32-bit register by the lanes where
// x < len (the predicate is formed in the same statement, so no register has to be zeroed or zero-extended)
template <typename T, int OFS>
__device__ __forceinline__ uint32_t i2_lds_lt(uint32_t sa, uint32_t x, uint32_t len) {
	uint32_t v;
	if (sizeof(T) == 1) {
		asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %1, %2;\n\t@p ld.shared.u8 %0, [%3+%4];\n\t}" : "=r"(v) : "r"(x), "r"(len), "r"(sa), "n"(OFS) : "memory");
	} else {
		asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %1, %2;\n\t@p ld.shared.u16 %0, [%3+%4];\n\t}" : "=r"(v) : "r"(x), "r"(len), "r"(sa), "n"(OFS) : "memory");
	}
	return v;
}
template <typename T, int OFS>
__device__ __forceinline__ void i2_sts_lt(uint32_t sa, uint32_t x, uint32_t len, uint32_t v) {
	if (sizeof(T) == 1) {
		asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %0, %1;\n\t@p st.shared.u8 [%2+%3], %4;\n\t}" ::"r"(x), "r"(len), "r"(sa), "n"(OFS), "r"(v) : "memory");
	} else {
		asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %0, %1;\n\t@p st.shared.u16 [%2+%3], %4;\n\t}" ::"r"(x), "r"(len), "r"(sa), "n"(OFS), "r"(v) : "memory");
	}
}

// a match of the common case (at most 64 elements, no overlap, neither range wraps around the ring): lane copies
// elements lane and lane + 32.  ring_sa: the ring's shared-memory byte address; d, s: those of element 0 of the
// destination (a ring slot) and of the source (ring or staging buffer, one index space: ring_sa + element index * sizeof(T))
template <int W, typename T>
__device__ __forceinline__ void i2_chk_simple(uint32_t ring_sa, uint32_t len, uint32_t d, uint32_t s) {
	constexpr uint32_t RING = W * sizeof(T), ALL = (W + 2u * I2Elem<T>::STAGE) * sizeof(T);
	const uint32_t dq = d - ring_sa, sq = s - ring_sa, n = len * (uint32_t)sizeof(T);
	OTZ_CHK(len == 0u || (dq + n <= RING && sq + n <= ALL && (sq >= RING || sq + n <= RING)), len && dq + n > RING ? OTZ_CK_LZ_RING_DST : OTZ_CK_LZ_RING_SRC);
}
template <typename T>
__device__ __forceinline__ void i2_copy_simple(uint32_t d, uint32_t s, uint32_t len, uint32_t lane) {
	// (d, s: addresses of element `lane`)
	const uint32_t v0 = i2_lds_lt<T, 0>(s, lane, len), v1 = i2_lds_lt<T, 32 * sizeof(T)>(s, lane + 32u, len);
	i2_sts_lt<T, 0>(d, lane, len, v0);
	i2_sts_lt<T, 32 * sizeof(T)>(d, lane + 32u, len, v1);
}

// what the scan of one batch leaves in registers for its execution
struct I2Batch {
	uint32_t ntake;     // records in the batch (0 = none left)
	uint32_t tot_l;     // literals it consumes
	uint32_t q_end;     // linear output position behind it
	uint32_t lr;        // this lane's record: literal run,
	uint32_t my_lit;    //   its first literal,
	uint32_t my_out;    //   its linear output position
	uint32_t lit4;      //   and its first four literal bytes
	// the match of this lane's record, as the executor wants it (it walks the records in stream order and fetches
	// these three words with one shuffle each):
	uint32_t mlen;      //   length | I2_MF_* flags above it: <= I2_ML_SIMPLE exactly when the match is the common case
	                    //   (length 0: no match)
	uint32_t mdst;      //   shared-memory byte address of the destination's ring slot
	uint32_t msrc;      //   shared-memory byte address of the source: a ring slot, or a slot of the staging buffer behind the
	                    //   ring (a FAR source, fetched while the batch before ran)
	uint32_t spec;      // warp-uniform: bit r set when record r is not the common case (mlen > I2_ML_SIMPLE)
};
#define I2_ML_LEN 0x1FFu          // mlen: the length
#define I2_ML_SIMPLE 64u          // at most 64 elements and no flag: two loads and two stores per lane, nothing else
#define I2_MF_DEP (1u << 9)       // the source reaches into what this batch itself writes
#define I2_MF_LONG (1u << 10)     // longer than 64 elements, or a range that wraps around the ring
#define I2_MF_PERIODIC (1u << 11) // distance < length

// scan records [b, b + 32) (this lane holds record b + lane in `rec`): positions by warp prefix sums, the match descriptor
// of every record (kept in its lane), and the copies of the batch's far sources into staging buffer `buf` are started.
// WIDE: 8-byte records {literal run | (length - 3) << 9, distance} (Zstandard: distances beyond 32 KiB); `rec` is the first
// word, `wdist` the second.  Otherwise the distance sits in rec[31:17].
template <int W, bool WIDE, typename T>
__device__ __forceinline__ I2Batch i2_scan_batch(I2LzSmem<W, T> &S, int buf, uint32_t rec, uint32_t wdist, uint32_t b, uint32_t nseq, uint32_t q,
	uint32_t lp, const uint8_t *__restrict__ lits, const T *gbase, uint32_t lane) {
	constexpr uint32_t MASK = I2Ring<W>::MASK, SPAN_MAX = I2Ring<W>::SPAN_MAX, VEC = I2Elem<T>::VEC, STAGE_VECS = I2Elem<T>::STAGE_VECS;
	const uint32_t lt_mask = (1u << lane) - 1u;
	I2Batch B;
	const bool have = b + lane < nseq;
	const uint32_t lr = have ? rec & 511u : 0u;
	const uint32_t ml = (have && lr != I2_SEQ_ESC) ? ((rec >> 9) & 255u) + 3u : 0u;
	const uint32_t dist = WIDE ? wdist : (rec >> 17) + 1u;
	uint32_t lsum = lr, osum = lr + ml;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) {
		const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, lsum, d), c = __shfl_up_sync(0xFFFFFFFFu, osum, d);
		if ((int)lane >= d) {
			lsum += a;
			osum += c;
		}
	}
	// the longest prefix of the batch whose output fits SPAN_MAX (one record is at most 769 bytes)
	const uint32_t fit = __ballot_sync(0xFFFFFFFFu, have && osum <= SPAN_MAX);
	B.ntake = __popc(fit);   // osum is monotonic, so `fit` is a prefix mask
	const uint32_t last = B.ntake ? B.ntake - 1u : 0u;
	B.tot_l = B.ntake ? __shfl_sync(0xFFFFFFFFu, lsum, last) : 0u;
	const uint32_t tot_o = B.ntake ? __shfl_sync(0xFFFFFFFFu, osum, last) : 0u;
	const bool mine = lane < B.ntake;
	B.lr = mine ? lr : 0u;
	B.my_lit = lp + lsum - lr;
	B.my_out = q + osum - lr - ml;
	B.q_end = q + tot_o;
	// the first literals of the run travel in a register
	B.lit4 = 0;
#pragma unroll
	for (int t = 0; t < 4; t++) {
		if ((uint32_t)t < B.lr) {
			B.lit4 |= (uint32_t)lits[B.my_lit + t] << (8 * t);
		}
	}
	// far: the source lies below the ring window [q_end - W, q_end) of this batch
	const uint32_t mq = B.my_out + lr;   // match destination
	const bool is_match = mine && ml != 0u;
	const bool is_far = is_match && dist > (uint32_t)W - (B.q_end - mq);
	const uint32_t far_m = __ballot_sync(0xFFFFFFFFu, is_far);
	const uint32_t src_lin = mq - dist;
	uint32_t mb = src_lin & MASK;   // the source as an element index from the ring's base (>= W: staging buffer)
	bool taken = mine;
	if (far_m) {
		// staging vectors per far match (the source is copied as whole 16-byte vectors)
		const uint32_t soff = src_lin & (VEC - 1u);
		const uint32_t nch = is_far ? (soff + ml + VEC - 1u) / VEC : 0u;
		uint32_t incl = nch;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, incl, d);
			if ((int)lane >= d) {
				incl += a;
			}
		}
		// the batch ends in front of the first record whose far source no longer fits the staging buffer (one match needs at
		// most 34 vectors, so the first record always stays): a source fetched directly from HBM inside the execution loop
		// would stall the whole warp for a memory round trip.  The far / near verdicts above used the longer batch's end —
		// conservative in both directions (a far source lies even further below the shorter batch's window, a near one still
		// inside the ring).
		const uint32_t over = __ballot_sync(0xFFFFFFFFu, mine && incl > STAGE_VECS);
		if (over) {
			B.ntake = (uint32_t)__ffs(over) - 1u;
			const uint32_t last2 = B.ntake - 1u;
			B.tot_l = __shfl_sync(0xFFFFFFFFu, lsum, last2);
			B.q_end = q + __shfl_sync(0xFFFFFFFFu, osum, last2);
			taken = lane < B.ntake;
			B.lr = taken ? B.lr : 0u;
		}
		if (is_far && taken) {
			const uint32_t cst = incl - nch;
			OTZ_CHK(VEC * cst + soff + ml <= I2Elem<T>::STAGE, OTZ_CK_LZ_STAGE);
			mb = (uint32_t)W + (uint32_t)buf * I2Elem<T>::STAGE + VEC * cst + soff;
			// every lane fetches the vectors of its own match (cp.async groups are per thread: the executor waits for
			// its own group and then syncs the warp)
			uint32_t sa = (uint32_t)__cvta_generic_to_shared(&S.stage[buf][VEC * cst]);
			const T *g = gbase + (src_lin & ~(VEC - 1u));
#pragma unroll 1
			for (uint32_t v = 0; v < nch; v++) {
				asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(g) : "memory");
				sa += 16u;
				g += VEC;
			}
		}
	}
	const bool has_match = is_match && taken;
	// LONG: more than 64 elements, or the destination / a ring source wraps around the ring
	const uint32_t flags = has_match ? (((ml > 64u || (mq & MASK) + ml > (uint32_t)W || (!is_far && (src_lin & MASK) + ml > (uint32_t)W)) ? I2_MF_LONG : 0u) |
		((!is_far && dist < ml) ? I2_MF_PERIODIC : 0u)) : 0u;
	// DEP: the source reaches into what this batch itself writes (earlier matches, its literal runs), so the executor has
	// to make the stores before it visible first; every other match only reads older ring data or its staged source and
	// runs back to back with its neighbours (no WAR either: a near source lies above q_end - W, a slot no store of this
	// batch touches)
	const uint32_t dep = (has_match && src_lin + ml > q) ? I2_MF_DEP : 0u;
	B.mlen = has_match ? ml | dep | flags : 0u;
	const uint32_t ring_sa = (uint32_t)__cvta_generic_to_shared(S.ring);
	B.mdst = ring_sa + (mq & MASK) * (uint32_t)sizeof(T);
	B.msrc = ring_sa + mb * (uint32_t)sizeof(T);
	B.spec = __ballot_sync(0xFFFFFFFFu, B.mlen > I2_ML_SIMPLE);
	asm volatile("cp.async.commit_group;" ::: "memory");
	return B;
}

// SEG: `list` holds huge streams; the tokens of a stream are the chain of segments k_seg_stitch accepted, walked by
// this warp.  PAR: the work items are single segments of such chains (seg.par_items), executed over 16-bit symbols
// into the symbol buffer `out` with the 32 KiB before the segment standing in as MARKERS (k_seg_window resolves them).
#define I2_LZ_PARAMS uint8_t *__restrict__ out, const otz_entry *__restrict__ ents, const uint32_t *__restrict__ list, uint32_t n_list, \
	uint32_t *__restrict__ work_counter, const uint8_t *__restrict__ scratch, const uint64_t *__restrict__ tok_ofs, \
	const I2TokRes *__restrict__ tokres, int32_t *__restrict__ status, uint32_t *__restrict__ produced_out, I2SegCtl seg, uint32_t k_first
#define I2_LZ_ARGS out, ents, list, n_list, work_counter, scratch, tok_ofs, tokres, status, produced_out, seg, k_first
template <int W, bool WIDE, bool SEG, bool PAR>
__device__ __forceinline__ void i2_inflate_lz(I2_LZ_PARAMS) {
	typedef typename I2ElemOf<PAR>::type T;
	static_assert(!PAR || (SEG && !WIDE), "PAR executes segments of DEFLATE streams");
	extern __shared__ __align__(16) uint8_t smem_raw[];
	constexpr uint32_t MASK = I2Ring<W>::MASK, SEGB = I2Ring<W>::SEG, SPAN_MAX = I2Ring<W>::SPAN_MAX, VEC = I2Elem<T>::VEC;
	const uint32_t lane = threadIdx.x & 31u;
	I2LzSmem<W, T> &S = reinterpret_cast<I2LzSmem<W, T> *>(smem_raw)[threadIdx.x >> 5];
	T *const rb = S.ring;
	// the ring's shared-memory byte address, and this lane's byte offset within a match's first 32 elements
	const uint32_t ring_sa = (uint32_t)__cvta_generic_to_shared(rb), lo = lane * (uint32_t)sizeof(T), lane32 = lane + 32u;
	if (PAR) {
		n_list = *seg.n_par;
	}
	for (;;) {
		uint32_t k = 0;
		if (lane == 0) {
			k = atomicAdd(work_counter, 1u);
		}
		k = __shfl_sync(0xFFFFFFFFu, k, 0) + (PAR ? 0u : k_first);   // (list slots [k_first, n_list); PAR: items of seg.par_items)
		if (k >= n_list) {
			break;
		}
		I2TokRes tr;
		uint32_t nsegs = 1, par_c = 0;
		if (PAR) {
			const uint32_t it = seg.par_items[k];
			k = it >> 16;        // from here on: the stream
			par_c = it & 0xFFFFu;
			tr.ok = 1;
			tr.status = 0;
			tr.nseq = tr.nlit = 0;
		} else if (SEG) {
			nsegs = seg.par[k] ? 0u : seg.nlive[k];
			tr.ok = nsegs != 0u;
			tr.status = seg.seg_status[k];
			tr.nseq = tr.nlit = 0;
		} else {
			tr = tokres[k];
		}
		if (!tr.ok) {
			continue;
		}
		const uint32_t ei = list[k];
		const otz_entry e = ents[ei];
		T *const dstp = PAR ? reinterpret_cast<T *>(out) + seg.sym_start[k * I2_MAXSEG + par_c] : reinterpret_cast<T *>(out + e.out_ofs);
		const uint32_t mis = (uint32_t)((reinterpret_cast<uint64_t>(dstp) / sizeof(T)) & (VEC - 1u));
		// PAR: linear position I2_PREWIN is the segment's first element; the markers sit below it
		T *const gbase = dstp - mis - (PAR ? I2_PREWIN : 0u);
		uint32_t q = mis + (PAR ? I2_PREWIN : 0u), qf = q;   // linear write position / position up to which HBM holds the data
#ifdef OTZ_BOUNDS_CHECK
		// (linear position behind the last element this work item may write)
		const uint32_t q_limit = q + (PAR ? seg.res[k * I2_MAXSEG + seg.live[k * I2_MAXSEG + par_c]].produced : e.uncomp_size);
#endif
		if (PAR) {
			// marker for the element m places before the segment: 256 + (I2_PREWIN - m).  HBM gets all the matches can
			// reach, the ring the part of them a near match can address.
			const uint32_t reach = min(seg.res[k * I2_MAXSEG + seg.live[k * I2_MAXSEG + par_c]].reach, (uint32_t)I2_PREWIN);
			for (uint32_t m = 1u + lane; m <= reach; m += 32) {
				const T v = (T)(256u + I2_PREWIN - m);
				gbase[q - m] = v;
				if (m <= (uint32_t)W) {
					rb[(q - m) & MASK] = v;
				}
			}
			__syncwarp();
		}
		for (uint32_t sgi = 0; sgi < nsegs; sgi++) {
			const uint8_t *lits;
			const uint32_t *seq_end;
			uint32_t nseq, nlit;
			if (SEG) {
				const I2SegRes *r_ = &seg.res[k * I2_MAXSEG + seg.live[k * I2_MAXSEG + (PAR ? par_c : sgi)]];
				lits = scratch + r_->scr_lo;
				seq_end = reinterpret_cast<const uint32_t *>(scratch + r_->scr_hi);
				nseq = r_->nseq;
				nlit = r_->nlit;
			} else {
				lits = scratch + tok_ofs[k];
				seq_end = reinterpret_cast<const uint32_t *>(scratch + tok_ofs[k + 1]);
				nseq = tr.nseq;
				nlit = tr.nlit;
			}
			uint32_t lp = 0, b = 0;       // literals / records consumed
			__syncwarp();
			// records b + lane (recA) and b + 32 + lane (recB); WIDE: their second words in offA / offB
			const uint2 *const seq_end2 = reinterpret_cast<const uint2 *>(seq_end);
			uint32_t recA = 0, recB = 0, offA = 0, offB = 0;
			if (WIDE) {
				if (lane < nseq) {
					const uint2 r = seq_end2[-1 - (int32_t)lane];
					recA = r.x;
					offA = r.y;
				}
				if (32u + lane < nseq) {
					const uint2 r = seq_end2[-33 - (int32_t)lane];
					recB = r.x;
					offB = r.y;
				}
			} else {
				recA = lane < nseq ? __ldcs(seq_end - 1 - lane) : 0u;
				recB = 32u + lane < nseq ? __ldcs(seq_end - 33 - lane) : 0u;
			}
			int buf = 0;
			I2Batch cur = i2_scan_batch<W, WIDE, T>(S, 0, recA, offA, 0u, nseq, q, lp, lits, gbase, lane);
			while (cur.ntake) {
				// ---- scan batch k+1 and start its far copies
				const uint32_t b2 = b + cur.ntake;
				{
					const uint32_t j = cur.ntake + lane;
					const uint32_t fromA = __shfl_sync(0xFFFFFFFFu, recA, j & 31u), fromB = __shfl_sync(0xFFFFFFFFu, recB, j & 31u);
					recA = j < 32u ? fromA : fromB;
					if (WIDE) {
						const uint32_t oA = __shfl_sync(0xFFFFFFFFu, offA, j & 31u), oB = __shfl_sync(0xFFFFFFFFu, offB, j & 31u);
						offA = j < 32u ? oA : oB;
						recB = offB = 0;
						if (b2 + 32u + lane < nseq) {
							const uint2 r = seq_end2[-33 - (int32_t)(b2 + lane)];
							recB = r.x;
							offB = r.y;
						}
					} else {
						recB = b2 + 32u + lane < nseq ? __ldcs(seq_end - 33 - (b2 + lane)) : 0u;
					}
				}
				const I2Batch nxt = i2_scan_batch<W, WIDE, T>(S, buf ^ 1, recA, offA, b2, nseq, cur.q_end, lp + cur.tot_l, lits, gbase, lane);
				// ---- execute batch k: its far sources have landed in stage[buf]
				asm volatile("cp.async.wait_group 1;" ::: "memory");
				__syncwarp();
				{
					// literal runs, all records at once
					const uint32_t n4 = min(cur.lr, 4u);
					for (uint32_t t = 0; t < n4; t++) {
						rb[(cur.my_out + t) & MASK] = (T)(uint8_t)(cur.lit4 >> (8u * t));
					}
#pragma unroll 1
					for (uint32_t t = 4; t < cur.lr; t++) {
						rb[(cur.my_out + t) & MASK] = lits[cur.my_lit + t];
					}
				}
				// the matches in stream order: three shuffles fetch a record's descriptor.  The common case — up to 64 elements, no
				// overlap, neither range wraps around the ring, no dependency on this batch's stores — is two loads and two stores
				// per lane at addresses the scan resolved.  Such records run back to back in pairs, the loads of both before their
				// stores (neither reads what the other writes, see DEP); the warp-uniform mask `spec` cuts the batch into runs of
				// them, and the record behind each run takes the side path.
#pragma unroll 1
				for (uint32_t r = 0, spec = cur.spec;; r++, spec &= spec - 1u) {
					const uint32_t end = spec ? (uint32_t)__ffs(spec) - 1u : cur.ntake;
#pragma unroll 1
					for (; r + 1u < end; r += 2u) {
						const uint32_t la = __shfl_sync(0xFFFFFFFFu, cur.mlen, r), lb = __shfl_sync(0xFFFFFFFFu, cur.mlen, r + 1u);
						const uint32_t da = __shfl_sync(0xFFFFFFFFu, cur.mdst, r), db = __shfl_sync(0xFFFFFFFFu, cur.mdst, r + 1u);
						const uint32_t sa = __shfl_sync(0xFFFFFFFFu, cur.msrc, r), sb = __shfl_sync(0xFFFFFFFFu, cur.msrc, r + 1u);
						i2_chk_simple<W, T>(ring_sa, la, da, sa);
						i2_chk_simple<W, T>(ring_sa, lb, db, sb);
						const uint32_t a0 = i2_lds_lt<T, 0>(sa + lo, lane, la), a1 = i2_lds_lt<T, 32 * sizeof(T)>(sa + lo, lane32, la);
						const uint32_t b0 = i2_lds_lt<T, 0>(sb + lo, lane, lb), b1 = i2_lds_lt<T, 32 * sizeof(T)>(sb + lo, lane32, lb);
						i2_sts_lt<T, 0>(da + lo, lane, la, a0);
						i2_sts_lt<T, 32 * sizeof(T)>(da + lo, lane32, la, a1);
						i2_sts_lt<T, 0>(db + lo, lane, lb, b0);
						i2_sts_lt<T, 32 * sizeof(T)>(db + lo, lane32, lb, b1);
					}
					if (r < end) {
						const uint32_t l = __shfl_sync(0xFFFFFFFFu, cur.mlen, r), d = __shfl_sync(0xFFFFFFFFu, cur.mdst, r),
							s = __shfl_sync(0xFFFFFFFFu, cur.msrc, r);
						i2_chk_simple<W, T>(ring_sa, l, d, s);
						i2_copy_simple<T>(d + lo, s + lo, l, lane);
						r++;
					}
					if (!spec) {
						break;
					}
					// record r: the side path
					const uint32_t ml = __shfl_sync(0xFFFFFFFFu, cur.mlen, r), d = __shfl_sync(0xFFFFFFFFu, cur.mdst, r),
						s = __shfl_sync(0xFFFFFFFFu, cur.msrc, r);
					const uint32_t len = ml & I2_ML_LEN;
					__syncwarp();   // earlier ring stores of this batch are visible to the loads below
					if (ml < I2_MF_LONG) {
						// DEP only: once those stores are visible, the common case
						i2_chk_simple<W, T>(ring_sa, len, d, s);
						i2_copy_simple<T>(d + lo, s + lo, len, lane);
						continue;
					}
					const uint32_t dq = (d - ring_sa) / (uint32_t)sizeof(T), bsrc = (s - ring_sa) / (uint32_t)sizeof(T);
					if (ml & I2_MF_PERIODIC) {
						// (a ring source below the destination: the distance is their distance around the ring)
						i2_copy_periodic<W, T>(rb, dq, bsrc, (dq - bsrc) & MASK, len, lane);
					} else {
						const uint32_t smask = bsrc >= (uint32_t)W ? 0xFFFFFFFFu : MASK;   // staged sources are not wrapped
#pragma unroll 1
						for (uint32_t x = lane; x < len; x += 32) {
							rb[(dq + x) & MASK] = rb[(bsrc + x) & smask];
						}
					}
				}
				b = b2;
				lp += cur.tot_l;
				q = cur.q_end;
				__syncwarp();
				const uint32_t qa = q & ~(SEGB - 1u);
				if (qa > qf) {
					OTZ_CHK(qa <= q_limit, OTZ_CK_LZ_FLUSH);
					i2_flush_range<W, T>(gbase, rb, qf, qa, lane);
					qf = qa;
					__syncwarp();
				}
				cur = nxt;
				buf ^= 1;
			}
			asm volatile("cp.async.wait_group 0;" ::: "memory");
			// literals after the last match
			while (lp < nlit) {
				const uint32_t n = min(nlit - lp, SPAN_MAX);
				for (uint32_t t = lane; t < n; t += 32) {
					rb[(q + t) & MASK] = lits[lp + t];
				}
				lp += n;
				q += n;
				__syncwarp();
				const uint32_t qa = q & ~(SEGB - 1u);
				if (qa > qf) {
					OTZ_CHK(qa <= q_limit, OTZ_CK_LZ_FLUSH);
					i2_flush_range<W, T>(gbase, rb, qf, qa, lane);
					qf = qa;
					__syncwarp();
				}
			}
		}   // segments
		if (q > qf) {
			OTZ_CHK(q <= q_limit, OTZ_CK_LZ_FLUSH);
			i2_flush_range<W, T>(gbase, rb, qf, q, lane);
		}
		if (!PAR && lane == 0) {
			status[ei] = tr.status;
			produced_out[ei] = e.uncomp_size;
		}
		__syncwarp();
	}
}

// The chain walk (SEG, not PAR) keeps more state across its loops; its big ring leaves room for 3 CTAs an SM, and the
// register budget that goes with it spares it a spill.  Every other instantiation keeps the compiler's own choice.
template <int W, bool WIDE, bool SEG, bool PAR = false>
__global__ typename std::enable_if<!SEG || PAR>::type __launch_bounds__(128) k_inflate_lz(I2_LZ_PARAMS) {
	i2_inflate_lz<W, WIDE, SEG, PAR>(I2_LZ_ARGS);
}
template <int W, bool WIDE, bool SEG, bool PAR = false>
__global__ typename std::enable_if<SEG && !PAR>::type __launch_bounds__(128, 3) k_inflate_lz(I2_LZ_PARAMS) {
	i2_inflate_lz<W, WIDE, SEG, PAR>(I2_LZ_ARGS);
}

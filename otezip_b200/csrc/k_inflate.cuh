// k_inflate.cuh — batched raw-DEFLATE (RFC 1951) decoder, one tile of G lanes per entry.
//
// Replaces inflateInit2/inflate/inflateEnd as driven by otezip_extract_entry
// (/root/reference/src/lib/otezip.c:503-529; decoder src/lib/deflate-dec.inc.c:547-831, abbreviated
// "dec" below).  The reference decodes a symbol by pulling one bit at a time and scanning all
// <=288 (length, code) pairs after every bit (dec:671-691, :743-764).  Here:
//   * the compressed bytes are fetched as coalesced 32-bit words, G words per load, one word per
//     lane; the 64-bit bit buffer is refilled by a tile shuffle from that register window
//     (the next window is already in flight while the current one is consumed);
//   * literal/length and distance codes are looked up in per-stream shared-memory tables
//     (9-bit / 8-bit roots with second-level tables for longer codes); an entry carries the code
//     length, the extra-bit count and the length / distance base, so a symbol costs one lookup;
//   * the most recent W output bytes live in a per-stream shared-memory ring: literals and LZ77 copies
//     touch only shared memory, completed 16*G-byte segments leave for HBM as coalesced 16-byte stores;
//   * LZ77 copies are performed by all G lanes (bytes are independent once the period
//     `distance` is taken into account, so no lane waits on another);
//   * dynamic-block tables are built cooperatively (counts with shared-memory atomics, canonical
//     order with match_any ranks, root fill in parallel).
// The decoder is a strict RFC 1951 decoder.  It also evaluates the reference's end-of-input rule
// (dec:811-816: Z_BUF_ERROR as soon as the last input byte has been loaded and the stream is not
// finished — SURVEY.md F1) and reports it as the OTZ_STF_REF_EOB flag, so the host library can
// reproduce the reference's accept/reject decision bit for bit.
//
// D64 = true instantiates the Deflate64 decoder (ZIP method 9, PKWARE's "enhanced deflate"; the tables of zlib's
// contrib/infback9/inftree9.c): a 64 KiB window, length symbol 285 = base 3 + 16 extra bits (lengths 3..65,538),
// distance symbols 30 / 31 = base 32,769 / 49,153 + 14 extra bits, HDIST up to 32.  Everything else is shared; the
// D64 = false instantiations are the DEFLATE decoder unchanged.
#pragma once
#include "otz_common.cuh"
#include "k_copy.cuh"

#define INF_LIT_ROOT 9
#define INF_DST_ROOT 8
#define INF_LIT_CAP 852   // zlib's proven bound for (286 symbols, root 9, max 15)
#define INF_DST_CAP 416   // >= 402, libdeflate's bound for (32 symbols, root 8, max 15)

// 32-bit table entry: [4:0] code bits consumed at this level (LINK: index bits of the second-level
// table, 0 = invalid code), [8:5] number of extra bits, [10:9] kind, [31:16] value — literal byte,
// length base, distance base or second-level offset.  Bases and extra-bit counts are the tables of
// dec:720-725 / dec:766-771, folded into the entry when the table is built.
#define INF_K_LIT 0u   // literal (or, in the distance table, a valid distance symbol)
#define INF_K_LEN 1u
#define INF_K_EOB 2u
#define INF_K_LINK 3u
#define INF_ENTRY(cb, xb, kind, value) ((uint32_t)(cb) | ((uint32_t)(xb) << 5) | ((uint32_t)(kind) << 9) | ((uint32_t)(value) << 16))
#define INF_INVALID INF_ENTRY(0u, 0u, INF_K_LINK, 0u)
#define INF_KIND(e) (((e) >> 9) & 3u)
// Deflate64 only: bit 11 adds 16 to the extra-bit count ([8:5] holds 0..15; symbol 285 needs 16)
#define INF_XB16 (1u << 11)
template <bool D64>
__device__ __forceinline__ uint32_t inf_extra_bits(uint32_t e) {
	return D64 ? ((e >> 5) & 15u) | ((e >> 7) & 16u) : (e >> 5) & 15u;
}

struct __align__(16) InflateSmem {
	uint32_t lit[INF_LIT_CAP];
	uint32_t dst[INF_DST_CAP];
	uint16_t sorted[288];
	uint8_t lens[320];
	uint32_t cnt[16];
	uint16_t offs[16];
	uint16_t run[16];
	uint16_t first[16];
	uint8_t pre[128];
};

__constant__ uint8_t c_cl_order[19] = { 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15 };  // dec:146-148

// ------------------------------------------------------------------------------------------------
// Bit reader.  Every lane carries an identical copy of a 64-bit window {hi:lo} of the stream and a bit
// offset `pos` into it; the next 32 stream bits are one funnel shift away (peek), consuming is one add
// (skip).  When pos reaches 32 the window slides by one word (norm); that word comes from a register
// window of G words spread over the lanes (tile shuffle), refilled by one coalesced load per G words
// with the following window already in flight.
template <int G>
struct BitReader {
	const uint32_t *words;   // aligned base of the current stream position
	uint32_t n_words;        // words available from `words`
	uint32_t win_base;       // word index of win_cur[lane 0]
	uint32_t win_cur, win_next;
	uint32_t widx;           // next word of the current window to hand out
	int32_t words_left;      // words not yet moved into {hi:lo} (negative once past the end)
	uint32_t pad_bits;       // bits in the last word that lie beyond the stream end
	uint32_t lo, hi, pos;

	__device__ __forceinline__ uint32_t load(uint32_t idx) const { return idx < n_words ? __ldg(words + idx) : 0u; }

	template <typename Tile>
	__device__ __forceinline__ uint32_t next_word(const Tile &tile) {
		const uint32_t w = tile.shfl(win_cur, widx);
		words_left--;
		if (++widx == G) {
			widx = 0;
			win_base += G;
			win_cur = win_next;
			win_next = load(win_base + G + tile.thread_rank());
		}
		return w;
	}
	template <typename Tile>
	__device__ __forceinline__ void init(const Tile &tile, const uint8_t *p, uint64_t nbytes) {
		const uint64_t a = reinterpret_cast<uint64_t>(p);
		const uint32_t skipb = (uint32_t)(a & 3);
		words = reinterpret_cast<const uint32_t *>(a - skipb);
		n_words = (uint32_t)((skipb + nbytes + 3) >> 2);
		pad_bits = (uint32_t)(((uint64_t)n_words << 5) - ((skipb + nbytes) << 3));
		win_base = 0;
		const int lane = tile.thread_rank();
		win_cur = load(lane);
		win_next = load(G + lane);
		widx = 0;
		words_left = (int32_t)n_words;
		lo = next_word(tile);
		hi = next_word(tile);
		pos = 8 * skipb;
	}
	// afterwards pos < 32: at least 33 bits can be peeked/skipped before the next norm
	template <typename Tile>
	__device__ __forceinline__ void norm(const Tile &tile) {
		if (pos >= 32) {
			lo = hi;
			hi = next_word(tile);
			pos -= 32;
		}
	}
	__device__ __forceinline__ uint32_t peek() const { return __funnelshift_r(lo, hi, pos); }   // needs pos < 32
	__device__ __forceinline__ void skip(uint32_t n) { pos += n; }
	// bits of the stream not yet consumed (negative: read past the end)
	__device__ __forceinline__ int64_t remaining_bits() const {
		return ((int64_t)words_left << 5) + 64 - (int64_t)pos - (int64_t)pad_bits;
	}
};

// Table entry of symbol s whose code takes cb bits at this table level.
template <bool D64>
__device__ __forceinline__ uint32_t inf_symbol_entry(uint32_t s, uint32_t cb, bool is_dist) {
	if (is_dist) {
		if (s >= 30 && !D64) {
			return INF_INVALID;  // fixed-table symbols 30/31 (dec:766-774 would index past dist_base)
		}
		if (s < 4) {
			return INF_ENTRY(cb, 0u, INF_K_LIT, 1u + s);
		}
		const uint32_t xb = (s - 2) >> 1;
		return INF_ENTRY(cb, xb, INF_K_LIT, 1u + ((2u + (s & 1u)) << xb));  // dec:766-771
	}
	if (s < 256) {
		return INF_ENTRY(cb, 0u, INF_K_LIT, s);
	}
	if (s == 256) {
		return INF_ENTRY(cb, 0u, INF_K_EOB, 0u);
	}
	if (s >= 286) {
		return INF_INVALID;  // dec:794-797
	}
	const uint32_t v = s - 257;
	if (v < 8) {
		return INF_ENTRY(cb, 0u, INF_K_LEN, 3u + v);
	}
	if (v == 28) {
		return D64 ? INF_ENTRY(cb, 0u, INF_K_LEN, 3u) | INF_XB16 : INF_ENTRY(cb, 0u, INF_K_LEN, 258u);
	}
	const uint32_t xb = (v - 4) >> 2;
	return INF_ENTRY(cb, xb, INF_K_LEN, 3u + ((4u + (v & 3u)) << xb));  // dec:720-725
}

// ------------------------------------------------------------------------------------------------
// Canonical table build from code lengths (dec:86-119 assigns the same canonical codes).
// Returns 0 ok, nonzero = invalid set.  All lanes return the same value.
template <int G, bool D64, typename Tile>
__device__ __noinline__ int build_table(const Tile &tile, InflateSmem &S, const uint8_t *lens, int n, int root, uint32_t *tbl, int cap,
	bool is_dist) {
	const int lane = tile.thread_rank();
	for (int i = lane; i < 16; i += G) {
		S.cnt[i] = 0;
	}
	tile.sync();
	for (int s = lane; s < n; s += G) {
		const uint32_t l = lens[s];
		if (l) {
			atomicAdd(&S.cnt[l], 1u);
		}
	}
	tile.sync();
	int left = 1, ncodes = 0, maxlen = 0;
	{
		int code = 0, off = 0;
		for (int l = 1; l <= 15; l++) {
			const int c = (int)S.cnt[l];
			left = (left << 1) - c;
			if (left < 0) {
				return 1;  // over-subscribed
			}
			code = (code + (l > 1 ? (int)S.cnt[l - 1] : 0)) << 1;
			if (lane == 0) {
				S.offs[l] = (uint16_t)off;
				S.run[l] = (uint16_t)off;
				S.first[l] = (uint16_t)code;
			}
			off += c;
			ncodes += c;
			if (c) {
				maxlen = l;
			}
		}
	}
	const int rootsz = 1 << root;
	if (ncodes == 0) {
		if (!is_dist) {
			return 1;
		}
		for (int k = lane; k < rootsz; k += G) {
			tbl[k] = INF_INVALID;  // a block of literals only: any distance code is an error
		}
		tile.sync();
		return 0;
	}
	if (left > 0) {
		if (!(ncodes == 1 && S.cnt[1] == 1)) {
			return 1;  // incomplete set (zlib accepts only a single 1-bit code)
		}
		for (int k = lane; k < rootsz; k += G) {
			tbl[k] = INF_INVALID;
		}
	}
	tile.sync();
	// canonical order: sorted[] = symbols by (length, symbol)
	for (int base = 0; base < n; base += G) {
		const int s = base + lane;
		const uint32_t l = s < n ? lens[s] : 0u;
		const uint32_t m = tile.match_any(l);
		const int rank = __popc(m & ((1u << lane) - 1u));
		if (l) {
			S.sorted[S.run[l] + rank] = (uint16_t)s;
		}
		tile.sync();
		if (l && rank == 0) {
			S.run[l] = (uint16_t)(S.run[l] + __popc(m));
		}
		tile.sync();
	}
	// root entries, one canonical index per lane
	for (int i = lane; i < ncodes; i += G) {
		const uint32_t s = S.sorted[i];
		const uint32_t l = lens[s];
		if ((int)l > root) {
			continue;
		}
		const uint32_t c = S.first[l] + (i - S.offs[l]);
		const uint32_t rev = __brev(c) >> (32 - l);
		const uint32_t e = inf_symbol_entry<D64>(s, l, is_dist);
		for (int k = (int)rev; k < rootsz; k += (1 << l)) {
			tbl[k] = e;
		}
	}
	// codes longer than the root: second-level tables, walked in canonical order by the whole tile
	if (maxlen > root) {
		int next_free = rootsz, cur_prefix = -1, sub_off = 0, sub_bits = 0;
		for (int i = S.offs[root + 1]; i < ncodes; i++) {
			const uint32_t s = S.sorted[i];
			const int l = lens[s];
			const uint32_t c = S.first[l] + (i - S.offs[l]);
			const uint32_t rev = __brev(c) >> (32 - l);
			const int prefix = (int)(rev & (uint32_t)(rootsz - 1));
			if (prefix != cur_prefix) {
				int curr = l - root;
				int lf = 1 << curr;
				int rem = (int)S.offs[l] + (int)S.cnt[l] - i;  // codes of this length still to place
				while (curr + root < maxlen) {
					lf -= rem;
					if (lf <= 0) {
						break;
					}
					curr++;
					lf <<= 1;
					rem = (int)S.cnt[curr + root];
				}
				if (next_free + (1 << curr) > cap) {
					return 1;  // cannot happen for a valid code (cap is the proven bound)
				}
				sub_off = next_free;
				sub_bits = curr;
				next_free += 1 << curr;
				cur_prefix = prefix;
				if (lane == 0) {
					tbl[prefix] = INF_ENTRY((uint32_t)sub_bits, 0u, INF_K_LINK, (uint32_t)sub_off);
				}
			}
			const uint32_t nb2 = (uint32_t)(l - root);
			const uint32_t e = inf_symbol_entry<D64>(s, nb2, is_dist);
			const int step = 1 << nb2;
			for (int k = (int)(rev >> root) + lane * step; k < (1 << sub_bits); k += G * step) {
				tbl[sub_off + k] = e;
			}
		}
	}
	tile.sync();
	return 0;
}

// dec:322-349
template <int G, bool D64, typename Tile>
__device__ __noinline__ int build_fixed(const Tile &tile, InflateSmem &S) {
	const int lane = tile.thread_rank();
	for (int i = lane; i < 320; i += G) {
		S.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5;
	}
	tile.sync();
	int r = build_table<G, D64>(tile, S, S.lens, 288, INF_LIT_ROOT, S.lit, INF_LIT_CAP, false);
	r |= build_table<G, D64>(tile, S, S.lens + 288, 32, INF_DST_ROOT, S.dst, INF_DST_CAP, true);
	return r;
}

// dec:122-266
template <int G, bool D64, typename Tile>
__device__ __forceinline__ int read_dynamic(const Tile &tile, InflateSmem &S, BitReader<G> &br) {
	const int lane = tile.thread_rank();
	br.norm(tile);
	uint32_t bits = br.peek();
	const int hlit = (int)(bits & 31) + 257, hdist = (int)((bits >> 5) & 31) + 1, hclen = (int)((bits >> 10) & 15) + 4;
	br.skip(14);
	if (hlit > 286 || (!D64 && hdist > 30)) {
		return 1;  // RFC 1951 limits; dec:165-168 would overflow its scratch instead (Deflate64: HDIST up to 32, lens[] holds 286 + 32)
	}
	for (int i = lane; i < 19; i += G) {
		S.lens[i] = 0;
	}
	tile.sync();
	uint64_t cnt = 0;  // packed byte counters, cnt>>(8*l) & 0xFF = number of precode symbols of length l
	for (int i = 0; i < hclen; i++) {
		br.norm(tile);
		const uint32_t v = br.peek() & 7u;
		br.skip(3);
		if (lane == 0) {
			S.lens[c_cl_order[i]] = (uint8_t)v;
		}
		cnt += 1ull << (8 * v);
	}
	tile.sync();
	// the code-length code must be complete (zlib: type CODES)
	uint64_t first = 0;  // packed first canonical code per length
	{
		int left = 1, code = 0;
		for (int l = 1; l <= 7; l++) {
			const int c = (int)((cnt >> (8 * l)) & 0xFF);
			left = (left << 1) - c;
			if (left < 0) {
				return 1;
			}
			code = (code + (l > 1 ? (int)((cnt >> (8 * (l - 1))) & 0xFF) : 0)) << 1;
			first |= (uint64_t)(code & 0xFF) << (8 * l);
		}
		if (left != 0) {
			return 1;
		}
	}
	for (int s = lane; s < 19; s += G) {
		const uint32_t l = S.lens[s];
		if (l) {
			int rank = 0;
			for (int t = 0; t < s; t++) {
				rank += (S.lens[t] == l);
			}
			const uint32_t c = (uint32_t)((first >> (8 * l)) & 0xFF) + rank;
			const uint32_t rev = __brev(c) >> (32 - l);
			for (uint32_t k = rev; k < 128; k += (1u << l)) {
				S.pre[k] = (uint8_t)(s | (l << 5));
			}
		}
	}
	tile.sync();
	// code lengths of the literal/length and distance alphabets (now overwrites S.lens)
	const int total = hlit + hdist;
	int idx = 0;
	uint32_t prev = 0;
	while (idx < total) {
		br.norm(tile);
		bits = br.peek();
		const uint32_t e = S.pre[bits & 127u];
		const uint32_t sym = e & 31u, cl = e >> 5;
		if (sym < 16) {
			br.skip(cl);
			if (lane == 0) {
				S.lens[idx] = (uint8_t)sym;
			}
			idx++;
			prev = sym;
			continue;
		}
		int rep;
		uint32_t val = 0;
		if (sym == 16) {  // dec:209-219
			if (idx == 0) {
				return 1;
			}
			val = prev;
			rep = 3 + (int)((bits >> cl) & 3u);
			br.skip(cl + 2);
		} else if (sym == 17) {  // dec:221-228
			rep = 3 + (int)((bits >> cl) & 7u);
			br.skip(cl + 3);
		} else {  // dec:230-237
			rep = 11 + (int)((bits >> cl) & 127u);
			br.skip(cl + 7);
		}
		if (idx + rep > total) {
			return 1;  // dec:244
		}
		for (int i = lane; i < rep; i += G) {
			S.lens[idx + i] = (uint8_t)val;
		}
		idx += rep;
		prev = val;
	}
	tile.sync();
	if (S.lens[256] == 0) {
		return 1;  // no end-of-block code
	}
	int r = build_table<G, D64>(tile, S, S.lens, hlit, INF_LIT_ROOT, S.lit, INF_LIT_CAP, false);
	if (r) {
		return r;
	}
	return build_table<G, D64>(tile, S, S.lens + hlit, hdist, INF_DST_ROOT, S.dst, INF_DST_CAP, true);
}

// ------------------------------------------------------------------------------------------------
// Output ring.  The last W bytes of a stream's output live in shared memory: literals are single
// byte stores by lane 0, LZ77 copies run ring -> ring (shared-memory latency instead of an L2 round
// trip per dependent copy), and every completed 16*G-byte segment goes to HBM as one coalesced
// 16-byte-per-lane store.  Ring index of output byte p is (p + mis) & (W-1) with mis = dst & 15, so ring
// vectors line up with 16-byte aligned global vectors.  A back-reference that reaches further than the ring
// holds is read from HBM (those bytes were flushed long ago: W >= 16*G + 516).
template <int G, int W>
struct __align__(16) InflateSmemV2 {
	InflateSmem t;
	uint8_t ring[W];
};

template <int G, int W>
struct OutRing {
	uint8_t *ring;
	uint8_t *gbase;     // dst - mis (16-byte aligned)
	uint32_t mis;
	uint32_t q;         // linear write position = bytes produced + mis
	uint32_t qf;        // linear position up to which HBM holds the data
	static constexpr uint32_t MASK = W - 1;
	static constexpr uint32_t SEG = 16 * G;

	__device__ __forceinline__ void init(uint8_t *r, uint8_t *dst) {
		ring = r;
		mis = (uint32_t)(reinterpret_cast<uint64_t>(dst) & 15);
		gbase = dst - mis;
		q = qf = mis;
	}
	__device__ __forceinline__ uint32_t produced() const { return q - mis; }
	// write ring[a, b) (linear positions) to HBM; whole tile, ring contents visible (caller synced)
	__device__ __forceinline__ void flush_range(uint32_t a, uint32_t b, int lane) {
		uint32_t a16 = (a + 15u) & ~15u, b16 = b & ~15u;
		if (a16 >= b16) {
			for (uint32_t x = a + lane; x < b; x += G) {
				gbase[x] = ring[x & MASK];
			}
			return;
		}
		for (uint32_t x = a + lane; x < a16; x += G) {
			gbase[x] = ring[x & MASK];
		}
		for (uint32_t x = a16 + 16u * lane; x < b16; x += SEG) {
			*reinterpret_cast<uint4 *>(gbase + x) = *reinterpret_cast<const uint4 *>(ring + (x & MASK));
		}
		for (uint32_t x = b16 + lane; x < b; x += G) {
			gbase[x] = ring[x & MASK];
		}
	}
	template <typename Tile>
	__device__ __forceinline__ void maybe_flush(const Tile &tile, int lane) {
		const uint32_t qa = q & ~(SEG - 1u);
		if (qa > qf) {
			tile.sync();
			flush_range(qf, qa, lane);
			qf = qa;
		}
	}
	template <typename Tile>
	__device__ __forceinline__ void finish(const Tile &tile, int lane) {
		tile.sync();
		if (q > qf) {
			flush_range(qf, q, lane);
			qf = q;
		}
	}
};

// LZ77 copy of length <= 258 bytes from `dist` bytes back to linear position dq (whole tile; dist already validated).
template <int G, int W, typename Tile>
__device__ __forceinline__ void inf_copy(const Tile &tile, const OutRing<G, W> &ring, uint8_t *rb, uint32_t dq, uint32_t dist, uint32_t length,
	int lane) {
	constexpr uint32_t MASK = W - 1;
	tile.sync();  // earlier ring stores of this tile are visible to the loads below
	if (dist + length <= (uint32_t)W) {
		const uint32_t sq = dq - dist;
		if (dist >= length) {
			for (uint32_t i = lane; i < length; i += G) {
				rb[(dq + i) & MASK] = rb[(sq + i) & MASK];
			}
		} else {
			// overlapping copy = periodic extension of the last `dist` bytes (dec:521-533)
			uint32_t r = dist > (uint32_t)lane ? (uint32_t)lane : (uint32_t)lane % dist;
			const uint32_t step = dist > (uint32_t)G ? (uint32_t)G : (uint32_t)G % dist;
			for (uint32_t i = lane; i < length; i += G) {
				rb[(dq + i) & MASK] = rb[(sq + r) & MASK];
				r += step;
				r = r >= dist ? r - dist : r;
			}
		}
	} else {
		// far back-reference: the source left the ring and is in HBM already (dist > W - 258 >= length)
		const uint8_t *sp = ring.gbase + (dq - dist);
		for (uint32_t i = lane; i < length; i += G) {
			rb[(dq + i) & MASK] = sp[i];
		}
	}
}

// One literal / end-of-block / length+distance step (dec:662-799).  CHECKED adds the tests that only matter
// near the end of the input or of the output buffer.  Returns 0 = continue, 1 = end of block, <0 = -status;
// Deflate64 only: 2 = a match longer than 258 bytes was executed (the caller's byte budget no longer holds).
template <int G, int W, bool CHECKED, bool D64, typename Tile>
__device__ __forceinline__ int inflate_event(const Tile &tile, const InflateSmem &S, BitReader<G> &br, OutRing<G, W> &ring, uint8_t *rb,
	uint32_t qcap, int lane) {
	constexpr uint32_t MASK = W - 1;
	uint32_t bits = br.peek();
	uint32_t e = S.lit[bits & ((1u << INF_LIT_ROOT) - 1u)];
	uint32_t cb = e & 31u;
	if (INF_KIND(e) == INF_K_LINK) {
		if (cb == 0) {
			return -OTZ_ST_DATA;  // dec:693-695: no code matches
		}
		e = S.lit[(e >> 16) + ((bits >> INF_LIT_ROOT) & ((1u << cb) - 1u))];
		if (INF_KIND(e) == INF_K_LINK) {
			return -OTZ_ST_DATA;
		}
		cb = (e & 31u) + INF_LIT_ROOT;
	}
	if (INF_KIND(e) == INF_K_LIT) {
		br.skip(cb);
		if (CHECKED && ring.q >= qcap) {
			return -OTZ_ST_OVERFLOW;  // dec:700-703
		}
		if (lane == 0) {
			rb[ring.q & MASK] = (uint8_t)(e >> 16);
		}
		ring.q++;
		return 0;
	}
	if (INF_KIND(e) == INF_K_EOB) {
		br.skip(cb);
		return 1;  // dec:711-716
	}
	// length (dec:720-737), then distance (dec:740-782)
	const uint32_t xb = inf_extra_bits<D64>(e);   // cb + xb <= 15 + 16: within the 32 peeked bits
	const uint32_t length = (e >> 16) + ((bits >> cb) & ((1u << xb) - 1u));
	br.skip(cb + xb);
	br.norm(tile);
	bits = br.peek();
	uint32_t d = S.dst[bits & ((1u << INF_DST_ROOT) - 1u)];
	uint32_t db = d & 31u;
	if (INF_KIND(d) == INF_K_LINK) {
		if (db == 0) {
			return -OTZ_ST_DATA;  // dec:762-764
		}
		d = S.dst[(d >> 16) + ((bits >> INF_DST_ROOT) & ((1u << db) - 1u))];
		if (INF_KIND(d) == INF_K_LINK) {
			return -OTZ_ST_DATA;
		}
		db = (d & 31u) + INF_DST_ROOT;
	}
	const uint32_t dxb = (d >> 5) & 15u;
	const uint32_t dist = (d >> 16) + ((bits >> db) & ((1u << dxb) - 1u));
	br.skip(db + dxb);
	const uint32_t dq = ring.q;
	if (dist > dq - ring.mis) {
		return -OTZ_ST_DATA;  // reaches before the start of the output (dec:785 does not check; strict)
	}
	if (CHECKED && length > qcap - dq) {
		return -OTZ_ST_OVERFLOW;  // dec:535-541, :791-793
	}
	if (D64 && length > 258u) {
		if (!CHECKED && length > qcap - dq) {
			return -OTZ_ST_OVERFLOW;
		}
		// A match of length L at distance d is the same as consecutive matches of <= 258 bytes, all at distance d.  Running
		// them as such, with the ring flush the event loop performs between events, keeps every invariant of the
		// 258-byte copy: the ring holds the pieces, a far source is already in HBM, overlap is the periodic copy.
		uint32_t q = dq, left = length;
		for (;;) {
			const uint32_t n = min(left, 258u);
			OTZ_CHK(q + n <= qcap, OTZ_CK_D64_OUT);
			OTZ_CHK(q - dist >= ring.mis && (dist + n <= (uint32_t)W || q - dist + n <= ring.qf), OTZ_CK_D64_SRC);
			inf_copy<G, W>(tile, ring, rb, q, dist, n, lane);
			q += n;
			left -= n;
			ring.q = q;
			if (!left) {
				break;
			}
			ring.maybe_flush(tile, lane);
		}
		return CHECKED ? 0 : 2;
	}
	inf_copy<G, W>(tile, ring, rb, dq, dist, length, lane);
	ring.q = dq + length;
	return 0;
}

// Decode one raw stream.  Returns the status word; *produced = bytes written.
template <int G, int W, bool D64, typename Tile>
__device__ __forceinline__ int32_t inflate_stream(const Tile &tile, InflateSmemV2<G, W> &SS, const uint8_t *__restrict__ in, uint32_t comp,
	uint8_t *__restrict__ out, uint32_t cap, uint32_t *produced, uint32_t row_flags) {
	const int lane = tile.thread_rank();
	InflateSmem &S = SS.t;
	*produced = 0;
	// a chunk row stops at the block boundary where its input ends (the last chunk at the stream's final block)
	const bool chunk_mid = (row_flags & OTZ_EF_CHUNK) && !(row_flags & OTZ_EF_LAST_CHUNK);
	if (comp == 0) {
		return OTZ_ST_TRUNCATED;  // dec:610: the loop never runs; Z_OK or Z_BUF_ERROR, never STREAM_END
	}
	BitReader<G> br;
	br.init(tile, in, comp);
	OutRing<G, W> ring;
	ring.init(SS.ring, out);
	uint8_t *const rb = SS.ring;
	constexpr uint32_t MASK = W - 1;
	const uint32_t qcap = cap + ring.mis;   // linear end of the output buffer
	bool ref_eob = false;
	int32_t err = 0;

// The reference returns Z_BUF_ERROR once ceil(bitpos/8) == comp while the stream is unfinished, i.e.
// fewer than 8 stream bits remain.  Only reachable when at most one word is left to load.
#define INF_STEP_CHECK()                                \
	if (br.words_left <= 1) {                           \
		const int64_t rem_ = br.remaining_bits();       \
		if (rem_ < 0) {                                 \
			err = OTZ_ST_TRUNCATED;                     \
			break;                                      \
		}                                               \
		if (rem_ < 8) {                                 \
			ref_eob = true;                             \
		}                                               \
	}

	for (;;) {
		// ---- block header, dec:613-627
		br.norm(tile);
		const uint32_t hdr = br.peek();
		const uint32_t final_blk = hdr & 1u;
		const uint32_t btype = (hdr >> 1) & 3u;
		br.skip(3);
		INF_STEP_CHECK();
		if (chunk_mid && final_blk) {
			// a chunk that is not the last one never holds the final block: the sequential decoder would stop here and
			// zero-pad the rest, so an index that says otherwise is wrong (the entry is then decoded as one stream)
			err = OTZ_ST_DATA;
			break;
		}
		if (btype == 0) {
			// ---- stored block, dec:269-319
			const int64_t rem = br.remaining_bits();
			const uint64_t pos = (uint64_t)comp - (uint64_t)(rem >> 3);  // partial byte dropped
			if ((uint64_t)comp - pos < 4) {
				err = OTZ_ST_DATA;
				break;
			}
			const uint32_t len = ld_le16(in + pos), nlen = ld_le16(in + pos + 2);
			if (len != ((~nlen) & 0xFFFFu) || (uint64_t)comp - pos - 4 < len) {
				err = OTZ_ST_DATA;
				break;
			}
			if (qcap - ring.q < len) {
				err = OTZ_ST_OVERFLOW;
				break;
			}
			const uint8_t *sp = in + pos + 4;
			for (uint32_t done = 0; done < len;) {
				const uint32_t n = min(len - done, OutRing<G, W>::SEG);
				for (uint32_t i = lane; i < n; i += G) {
					rb[(ring.q + i) & MASK] = sp[done + i];
				}
				ring.q += n;
				done += n;
				ring.maybe_flush(tile, lane);
			}
			const uint64_t npos = pos + 4 + len;
			br.init(tile, in + npos, (uint64_t)comp - npos);
			if (final_blk) {
				break;
			}
			if (npos >= comp) {  // dec:811-816 after a non-final stored block
				if (chunk_mid) {
					break;   // end of this chunk
				}
				ref_eob = true;
			}
			continue;
		}
		if (btype == 3) {
			err = OTZ_ST_DATA;  // dec:657-658
			break;
		}
		if ((btype == 1 ? build_fixed<G, D64>(tile, S) : read_dynamic<G, D64>(tile, S, br)) != 0) {
			err = OTZ_ST_DATA;
			break;
		}
		INF_STEP_CHECK();
		// ---- symbols.  An event consumes at most 48 bits (Deflate64: 60; two window words) and produces at most 258 bytes, so
		// `budget` events can run without any end-of-input / end-of-output test; the rest run one by one.  (A longer Deflate64
		// match tests the end of the output itself and ends the run of unchecked events.)
		bool eob = false;
		for (;;) {
			int64_t budget = min(((int64_t)br.words_left - 2) >> 1, (int64_t)((qcap - ring.q) / 258u));
			budget = min(budget, (int64_t)1 << 20);
			int rc = 0;
			for (int32_t n = (int32_t)budget; n > 0; n--) {
				br.norm(tile);
				rc = inflate_event<G, W, false, D64>(tile, S, br, ring, rb, qcap, lane);
				if (rc) {
					break;
				}
				ring.maybe_flush(tile, lane);
			}
			if (D64 && rc == 2) {
				ring.maybe_flush(tile, lane);
				continue;   // a long match used up an unknown part of the byte budget: compute it again
			}
			if (rc == 0 && budget <= 0) {
				br.norm(tile);
				rc = inflate_event<G, W, true, D64>(tile, S, br, ring, rb, qcap, lane);
				if (rc == 0) {
					ring.maybe_flush(tile, lane);
					INF_STEP_CHECK();
				}
			}
			if (rc > 0) {
				eob = true;
				break;
			}
			if (rc < 0) {
				err = -rc;
				break;
			}
		}
		if (err) {
			break;
		}
		if (!eob) {
			break;  // INF_STEP_CHECK left the loop with err set
		}
		if (final_blk) {
			if (br.remaining_bits() < 0) {
				err = OTZ_ST_TRUNCATED;
			}
			break;  // dec:714-716
		}
		// (a chunk that is not the last one ends only behind an empty stored block, byte aligned, exactly where its input
		// ends — the shape k_deflate writes; a Huffman block that merely runs out of input is not a chunk boundary: the
		// sequential decoder would read the next header from the bits left over)
		INF_STEP_CHECK();
	}
#undef INF_STEP_CHECK
	ring.finish(tile, lane);
	const uint32_t op = ring.produced();
	*produced = op;
	if (err) {
		return err;
	}
	if (row_flags & OTZ_EF_CHUNK) {
		return op == cap ? OTZ_ST_OK : OTZ_ST_SIZE;   // a chunk must fill its slice exactly
	}
	return OTZ_ST_OK | (ref_eob ? OTZ_STF_REF_EOB : 0) | (op < cap ? OTZ_STF_SHORT : 0);
}

// grid: persistent; each tile pulls the next entry of `list` (largest first) from a global counter.
// n_list_dev != NULL: the list length lives in device memory (written by an earlier kernel of the same stream).
template <int G, int W, bool D64 = false>
__global__ void __launch_bounds__(256) k_inflate(const uint8_t *__restrict__ archive, uint8_t *__restrict__ out,
	const otz_entry *__restrict__ ents, const OtzEntryState *__restrict__ est, int32_t *__restrict__ status,
	const uint32_t *__restrict__ list, uint32_t n_list, uint32_t *__restrict__ work_counter, uint32_t *__restrict__ produced_out,
	const uint32_t *__restrict__ n_list_dev) {
	extern __shared__ __align__(16) uint8_t smem_raw[];
	if (n_list_dev) {
		n_list = *n_list_dev;   // list filled on the device (fallback list of k_inflate_tok)
	}
	auto tile = cg::tiled_partition<G>(cg::this_thread_block());
	const int lane = tile.thread_rank();
	InflateSmemV2<G, W> &S = reinterpret_cast<InflateSmemV2<G, W> *>(smem_raw)[threadIdx.x / G];
	for (;;) {
		uint32_t k = 0;
		if (lane == 0) {
			k = atomicAdd(work_counter, 1u);
		}
		k = tile.shfl(k, 0);
		if (k >= n_list) {
			break;
		}
		const uint32_t ei = list[k];
		if (OTZ_ST_CODE(status[ei]) != OTZ_ST_OK) {
			continue;
		}
		const otz_entry e = ents[ei];
		uint8_t *dst = out + e.out_ofs;
		uint32_t produced = 0;
		int32_t st = inflate_stream<G, W, D64>(tile, S, archive + est[ei].data_ofs, e.comp_size, dst, e.uncomp_size, &produced, e.flags);
		if (D64 && OTZ_ST_CODE(st) == OTZ_ST_OK) {
			st |= OTZ_STF_REF_EOB;   // a valid stream of a method the reference rejects (otezip.c:662-665)
		}
		if ((e.flags & OTZ_EF_CHUNK) && OTZ_ST_CODE(st) != OTZ_ST_OK && lane == 0) {
			status[e.crc32] = OTZ_ST_DATA;   // a failing chunk fails its parent row (e.crc32 = parent row)
		}
		if (OTZ_ST_CODE(st) == OTZ_ST_OK && produced < e.uncomp_size) {
			// otezip.c:500 pre-zeroes the buffer and never compares total_out: short streams are zero-padded
			for (uint64_t i = (uint64_t)produced + lane; i < e.uncomp_size; i += G) {
				dst[i] = 0;
			}
		}
		if (lane == 0) {
			status[ei] = st;
			produced_out[ei] = produced;
		}
		tile.sync();
	}
}

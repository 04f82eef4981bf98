// k_xz.cuh — XZ entries (ZIP method 95): the xz container, LZMA2 chunks and the LZMA decoder.
//
// tests/xzref.py is the readable restatement of what these kernels do; the verdicts are its verdicts.
//
// k_xz_walk: one lane per XZ entry.  It parses the container (stream header, block headers, index, footer, stream padding)
// and hops the LZMA2 chunk headers without decoding them: every chunk header carries its packed and unpacked sizes.  It
// validates everything structural (CRC32s of the headers, index and footer; index against the blocks; the LZMA2 control
// and property rules; output beyond uncomp_size) and stops at the first error.  Every dictionary reset (the first chunk of a
// block, control 0x01, control >= 0xE0) starts a stream that depends on nothing before it; the walk cuts the entry into
// segments there, merging a reset into the running segment while that segment holds less than XZ_SEG_MIN bytes.  Each
// segment goes to the entry's slot range of the segment table, in stream order.
//
// k_lzma: one warp per segment, persistent grid, segments pulled from an atomic counter in walk order.  Lane 0 runs the
// range decoder over the probability model in shared memory and writes literals and short in-ring matches into the
// shared-memory output ring (OutRing of k_inflate.cuh).  The warp flushes the ring as coalesced 16-byte stores, executes
// long and far matches (inf_copy: far sources come from the entry's bytes in HBM, which are the dictionary), initialises the
// model on a reset and copies uncompressed chunks.  A segment that crosses a block or stream boundary hops the container
// structure without checking it again (the walk did).  Two shared-memory classes: lc + lp <= 3 (every xz preset) and
// lc + lp = 4, whose literal table is twice as large.
//
// k_xz_finish merges the verdicts: the first failing segment in stream order, else the walk's verdict, else OK.
#pragma once
#include "otz_common.cuh"
#include "k_inflate.cuh"

// A dictionary reset starts a new segment only once the running one holds this many bytes; the plan sizes the segment
// table from it (one slot per XZ_SEG_MIN bytes of declared output, plus one per entry).
#define XZ_SEG_MIN (16u * 1024u)
#define XZ_RING 4096u                   // output ring per warp
#define XZ_LANE0_MAX 16u                // matches at most this long, with their source in the ring, are copied by lane 0
#define XZ_NO_SEG 0xFFFFFFFFu

// probability model layout (tests/xzref.py: P_*)
#define XZ_P_ISMATCH 0
#define XZ_P_ISREP 192
#define XZ_P_ISREP0 204
#define XZ_P_ISREP1 216
#define XZ_P_ISREP2 228
#define XZ_P_ISREP0L 240
#define XZ_P_SLOT 432
#define XZ_P_SPEC 688
#define XZ_P_ALIGN 803
#define XZ_P_LEN 819
#define XZ_P_REPLEN 1333
#define XZ_P_LIT 1847
#define XZ_LEN_LOW 2
#define XZ_LEN_MID 130
#define XZ_LEN_HIGH 258

// One segment: a run of LZMA2 chunks that starts at a dictionary reset.  Offsets are relative to the entry's payload
// (input) and to its output slice.
struct XzSeg {
	uint32_t k;          // slot of the entry in the XZ work list; XZ_NO_SEG = empty slot
	uint32_t in_ofs;     // control byte of the first chunk
	uint32_t out_ofs;
	uint32_t out_bytes;
	uint32_t dict;       // dictionary size of the first chunk's block
	uint32_t meta;       // [7:0] largest lc + lp of the segment, [15:8] check bytes of the first chunk's stream
	uint32_t made;       // k_lzma, on an error: the bytes the segment produced before it
};

// Per XZ entry (one per work-list slot).
struct XzEnt {
	uint32_t first, cap;          // slot range of the segment table (plan)
	int32_t walk_st;              // the walk's verdict (OTZ_ST_OK when the whole container is valid)
	uint32_t walk_out;            // bytes the walked chunks declare
	unsigned long long err;       // (slot << 8) | status of the first failing segment; ~0 = none
};

__device__ __forceinline__ uint32_t xz_check_bytes(uint32_t id) {
	return id == 0 ? 0u : id == 1 ? 4u : id == 4 ? 8u : id == 10 ? 32u : 0xFFFFFFFFu;   // other IDs are reserved
}
__device__ __forceinline__ uint32_t xz_dict_size(uint32_t code) {
	return code == 40 ? 0xFFFFFFFFu : (2u | (code & 1u)) << (code / 2u + 11u);
}
__device__ __forceinline__ uint32_t xz_crc(const uint32_t *__restrict__ t0, uint32_t c, const uint8_t *p, uint32_t n) {
	for (uint32_t i = 0; i < n; i++) {
		c = t0[(c ^ p[i]) & 0xFFu] ^ (c >> 8);
	}
	return c;
}

// ------------------------------------------------------------------------------------------------ walk
// Unpadded size (header + compressed data + check) and unpacked size of the block at p, a block the walk has validated;
// returns the offset behind it.
__device__ __forceinline__ uint32_t xz_block_sizes(const uint8_t *in, uint32_t p, uint32_t csize, uint64_t &unpadded, uint64_t &unc) {
	uint32_t x = p + (in[p] + 1u) * 4u;
	unc = 0;
	for (;;) {
		const uint32_t c = in[x];
		if (c == 0) {
			x++;
			break;
		}
		if (c >= 0x80) {
			unc += ((c & 0x1Fu) << 16) + (in[x + 1] << 8) + in[x + 2] + 1u;
			x += (c >= 0xC0 ? 6u : 5u) + (in[x + 3] << 8) + in[x + 4] + 1u;
		} else {
			const uint32_t u = (in[x + 1] << 8) + in[x + 2] + 1u;
			unc += u;
			x += 3u + u;
		}
	}
	unpadded = (uint64_t)(x - p) + csize;
	return p + ((x - p + 3u) & ~3u) + csize;
}

// bounded reader of one payload; every failure leaves `st` set
struct XzRd {
	const uint8_t *in;
	uint32_t n, p;
	int32_t st;
	__device__ __forceinline__ bool need(uint32_t k) {
		if ((uint64_t)p + k > n) {
			st = OTZ_ST_TRUNCATED;
			return false;
		}
		return true;
	}
	__device__ __forceinline__ uint32_t byte() { return need(1) ? in[p++] : 0u; }
	// xz variable-length integer (at most 9 bytes, shortest encoding)
	__device__ __forceinline__ uint64_t vli() {
		uint64_t v = 0;
		for (int i = 0; i < 9; i++) {
			const uint32_t b = byte();
			if (st) {
				return 0;
			}
			v |= (uint64_t)(b & 0x7Fu) << (7 * i);
			if (!(b & 0x80u)) {
				if (b == 0 && i > 0) {
					st = OTZ_ST_DATA;
				}
				return v;
			}
		}
		st = OTZ_ST_DATA;
		return 0;
	}
};

__global__ void __launch_bounds__(128) k_xz_walk(const uint8_t *__restrict__ archive, const otz_entry *__restrict__ ents,
	const OtzEntryState *__restrict__ est, const int32_t *__restrict__ status, const uint32_t *__restrict__ list, uint32_t n_list,
	XzEnt *__restrict__ xe, XzSeg *__restrict__ segs, const uint32_t *__restrict__ t0, uint32_t *__restrict__ n_class) {
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= n_list) {
		return;
	}
	const uint32_t ei = list[k];
	const XzEnt me = xe[k];
	uint32_t nseg = 0;
	uint64_t out = 0;
	const otz_entry e = ents[ei];
	XzRd r{ archive + est[ei].data_ofs, e.comp_size, 0u, OTZ_ST_OK };
	// the running segment
	bool open = false;
	XzSeg cur{};
	auto close = [&]() {
		if (open && out > cur.out_ofs) {
			cur.out_bytes = (uint32_t)(out - cur.out_ofs);
			OTZ_CHK(nseg < me.cap, OTZ_CK_XZ_SEG);
			if (nseg < me.cap) {
				segs[me.first + nseg] = cur;
				atomicAdd(&n_class[(cur.meta & 0xFFu) > 3u], 1u);
			}
			nseg++;
		}
		open = false;
	};
	if (OTZ_ST_CODE(status[ei]) != OTZ_ST_OK) {
		r.st = status[ei];   // resolve failed: nothing to decode, the status stays
		goto done;
	}
	if (e.comp_size == 0) {
		r.st = OTZ_ST_TRUNCATED;
		goto done;
	}
	for (;;) {
		// ---- stream header
		if (!r.need(12)) {
			goto done;
		}
		const uint8_t *h = r.in + r.p;
		if (h[0] != 0xFD || h[1] != '7' || h[2] != 'z' || h[3] != 'X' || h[4] != 'Z' || h[5] != 0 ||
			~xz_crc(t0, ~0u, h + 6, 2) != ld_le32(h + 8) || h[6] != 0 || (h[7] & 0xF0u) || xz_check_bytes(h[7]) == 0xFFFFFFFFu) {
			r.st = OTZ_ST_DATA;
			goto done;
		}
		const uint32_t flags = ld_le16(h + 6), csize = xz_check_bytes(h[7]);
		r.p += 12;
		const uint32_t first_blk = r.p;
		uint32_t nblk = 0;
		for (;;) {
			const uint32_t hstart = r.p;
			const uint32_t b0 = r.byte();
			if (r.st) {
				goto done;
			}
			if (b0 == 0) {
				break;   // index indicator
			}
			// ---- block header
			const uint32_t hsize = (b0 + 1u) * 4u;
			if (!r.need(hsize - 1u)) {
				goto done;
			}
			if (~xz_crc(t0, ~0u, r.in + hstart, hsize - 4u) != ld_le32(r.in + hstart + hsize - 4u)) {
				r.st = OTZ_ST_DATA;
				goto done;
			}
			const uint32_t hend = hstart + hsize - 4u;
			const uint32_t bf = r.byte();
			const uint64_t hcomp = (bf & 0x40u) ? r.vli() : ~0ull, hunc = (bf & 0x80u) ? r.vli() : ~0ull;
			const uint64_t fid = r.vli(), npr = r.vli();
			if (r.st) {
				goto done;
			}
			if ((bf & 0x3Cu) || r.p + npr > hend) {
				r.st = OTZ_ST_DATA;
				goto done;
			}
			if ((bf & 3u) != 0 || fid != 0x21) {
				r.st = OTZ_ST_METHOD;   // a filter chain other than one LZMA2 filter: not on this path
				goto done;
			}
			const uint32_t prop = npr >= 1 ? r.in[r.p] : 0xFFu;
			if (npr != 1 || prop > 40 || hcomp == 0) {
				r.st = OTZ_ST_DATA;
				goto done;
			}
			for (uint32_t x = r.p + 1; x < hend; x++) {
				if (r.in[x]) {
					r.st = OTZ_ST_DATA;   // header padding
					goto done;
				}
			}
			const uint32_t dict = xz_dict_size(prop);
			r.p = hstart + hsize;
			// ---- LZMA2 chunks
			const uint32_t dstart = r.p;
			uint64_t bunc = 0;
			bool need_dict = true, need_props = true;
			for (;;) {
				const uint32_t cpos = r.p;
				const uint32_t c = r.byte();
				if (r.st) {
					goto done;
				}
				if (c == 0) {
					break;
				}
				const bool reset = c == 1 || c >= 0xE0;
				if (reset) {
					need_dict = false;
					need_props = true;
				} else if (need_dict || (c > 2 && c < 0x80)) {
					r.st = OTZ_ST_DATA;
					goto done;
				}
				uint32_t unp, pk, lclp = 0;
				if (c >= 0x80) {
					if (!r.need(4)) {
						goto done;
					}
					unp = ((c & 0x1Fu) << 16) + (r.in[r.p] << 8) + r.in[r.p + 1] + 1u;
					pk = (r.in[r.p + 2] << 8) + r.in[r.p + 3] + 1u;
					r.p += 4;
					if (c >= 0xC0) {
						const uint32_t pr = r.byte();
						if (r.st) {
							goto done;
						}
						lclp = pr % 9u + pr / 9u % 5u;
						if (pr > 224 || lclp > 4) {
							r.st = OTZ_ST_DATA;
							goto done;
						}
						need_props = false;
					} else if (need_props) {
						r.st = OTZ_ST_DATA;
						goto done;
					}
				} else {
					if (!r.need(2)) {
						goto done;
					}
					unp = pk = (r.in[r.p] << 8) + r.in[r.p + 1] + 1u;
					r.p += 2;
				}
				if (out + unp > e.uncomp_size) {
					r.st = OTZ_ST_OVERFLOW;
					goto done;
				}
				if (!r.need(pk)) {
					goto done;
				}
				if (reset && (!open || out - cur.out_ofs >= XZ_SEG_MIN)) {
					close();
					open = true;
					cur = XzSeg{ k, cpos, (uint32_t)out, 0u, dict, csize << 8, 0u };
				}
				cur.meta = max(cur.meta & 0xFFu, lclp) | (cur.meta & ~0xFFu);
				r.p += pk;
				out += unp;
				bunc += unp;
			}
			const uint32_t bcomp = r.p - dstart;
			if ((hcomp != ~0ull && hcomp != bcomp) || (hunc != ~0ull && hunc != bunc)) {
				r.st = OTZ_ST_DATA;
				goto done;
			}
			while ((r.p - hstart) & 3u) {
				const uint32_t pad = r.byte();
				if (r.st || pad) {
					r.st = r.st ? r.st : OTZ_ST_DATA;   // block padding
					goto done;
				}
			}
			if (!r.need(csize)) {
				goto done;
			}
			r.p += csize;   // the check field: skipped, the ZIP CRC-32 covers the entry
			nblk++;
		}
		// ---- index: the records must be those of the blocks, compared one by one with a second pass over the (validated)
		// blocks of this stream
		const uint32_t istart = r.p - 1u;
		const uint64_t cnt = r.vli();
		if (!r.st && cnt != nblk) {
			r.st = OTZ_ST_DATA;
		}
		for (uint32_t i = 0, bp = first_blk; i < nblk && !r.st; i++) {
			const uint64_t unpadded = r.vli(), unc = r.vli();
			uint64_t b_unpadded, b_unc;
			bp = xz_block_sizes(r.in, bp, csize, b_unpadded, b_unc);
			if (!r.st && (unpadded != b_unpadded || unc != b_unc)) {
				r.st = OTZ_ST_DATA;
			}
		}
		if (r.st) {
			goto done;
		}
		while ((r.p - istart) & 3u) {
			const uint32_t pad = r.byte();
			if (r.st || pad) {
				r.st = r.st ? r.st : OTZ_ST_DATA;
				goto done;
			}
		}
		if (!r.need(4)) {
			goto done;
		}
		if (~xz_crc(t0, ~0u, r.in + istart, r.p - istart) != ld_le32(r.in + r.p)) {
			r.st = OTZ_ST_DATA;
			goto done;
		}
		r.p += 4;
		// ---- footer
		if (!r.need(12)) {
			goto done;
		}
		{
			const uint8_t *f = r.in + r.p;
			if (~xz_crc(t0, ~0u, f + 4, 6) != ld_le32(f) || f[10] != 'Y' || f[11] != 'Z' || ld_le16(f + 8) != flags ||
				((uint64_t)ld_le32(f + 4) + 1u) * 4u != r.p - istart) {
				r.st = OTZ_ST_DATA;
				goto done;
			}
			r.p += 12;
		}
		// ---- stream padding (zero bytes, a multiple of 4), then the end or another stream
		const uint32_t z = r.p;
		while (r.p < r.n && r.in[r.p] == 0) {
			r.p++;
		}
		if ((r.p - z) & 3u) {
			r.st = OTZ_ST_DATA;
			goto done;
		}
		if (r.p == r.n) {
			break;
		}
	}
done:
	close();
	for (uint32_t s = nseg; s < me.cap; s++) {
		segs[me.first + s].k = XZ_NO_SEG;
	}
	xe[k].walk_st = r.st;
	xe[k].walk_out = (uint32_t)out;
	xe[k].err = ~0ull;
}

// ------------------------------------------------------------------------------------------------ decode
// Lane 0 -> warp requests
#define XZ_ACT_FLUSH 0
#define XZ_ACT_COPY 1    // a0 = distance (>= 1), a1 = length
#define XZ_ACT_INIT 2    // a0 = probabilities to set to 1024
#define XZ_ACT_RAW 3     // a0 = input offset, a1 = length: an uncompressed chunk
#define XZ_ACT_DONE 4
#define XZ_ACT_ERR 5

template <int LCLP>
struct XzSmem {
	static constexpr uint32_t NPROB = XZ_P_LIT + (0x300u << LCLP);
	uint8_t ring[XZ_RING];
	uint16_t probs[(NPROB + 7u) & ~7u];
};
// both classes fit the default dynamic shared-memory limit, so the launches need no attribute
static_assert(sizeof(XzSmem<4>) <= 48u * 1024u, "k_lzma<4> needs cudaFuncAttributeMaxDynamicSharedMemorySize");

// Bit of the adaptive binary model (LZMA's range decoder).  The input is the chunk's packed bytes [ip, iend): reads past
// the end see zero and only move ip, which the end-of-chunk test rejects.
#define XZ_NORM()                                              \
	if (range < (1u << 24)) {                                  \
		range <<= 8;                                           \
		code = (code << 8) | (ip < iend ? (uint32_t)in[ip] : 0u); \
		ip++;                                                  \
	}
#define XZ_BIT(idx, bitvar)                                    \
	do {                                                       \
		const uint32_t ix_ = (idx);                            \
		OTZ_CHK(ix_ < S.NPROB, OTZ_CK_XZ_PROB);                \
		XZ_NORM();                                             \
		const uint32_t pr_ = P[ix_];                           \
		const uint32_t bd_ = (range >> 11) * pr_;              \
		if (code < bd_) {                                      \
			range = bd_;                                       \
			P[ix_] = (uint16_t)(pr_ + ((2048u - pr_) >> 5));   \
			bitvar = 0;                                        \
		} else {                                               \
			range -= bd_;                                      \
			code -= bd_;                                       \
			P[ix_] = (uint16_t)(pr_ - (pr_ >> 5));             \
			bitvar = 1;                                        \
		}                                                      \
	} while (0)

template <int LCLP>
__device__ __forceinline__ uint32_t xz_tree(uint16_t *P, const XzSmem<LCLP> &S, uint32_t base, int nbits, uint32_t &range, uint32_t &code,
	uint32_t &ip, uint32_t iend, const uint8_t *in) {
	uint32_t m = 1;
	for (int i = 0; i < nbits; i++) {
		uint32_t b;
		XZ_BIT(base + m, b);
		m = (m << 1) | b;
	}
	return m - (1u << nbits);
}
template <int LCLP>
__device__ __forceinline__ uint32_t xz_rtree(uint16_t *P, const XzSmem<LCLP> &S, uint32_t base, int nbits, uint32_t &range, uint32_t &code,
	uint32_t &ip, uint32_t iend, const uint8_t *in) {
	uint32_t m = 1, v = 0;
	for (int i = 0; i < nbits; i++) {
		uint32_t b;
		XZ_BIT(base + m, b);
		m = (m << 1) | b;
		v |= b << i;
	}
	return v;
}
template <int LCLP>
__device__ __forceinline__ uint32_t xz_len(uint16_t *P, const XzSmem<LCLP> &S, uint32_t base, uint32_t ps, uint32_t &range, uint32_t &code,
	uint32_t &ip, uint32_t iend, const uint8_t *in) {
	uint32_t b;
	XZ_BIT(base, b);
	if (!b) {
		return 2u + xz_tree<LCLP>(P, S, base + XZ_LEN_LOW + ps * 8u - 1u, 3, range, code, ip, iend, in);
	}
	XZ_BIT(base + 1u, b);
	if (!b) {
		return 10u + xz_tree<LCLP>(P, S, base + XZ_LEN_MID + ps * 8u - 1u, 3, range, code, ip, iend, in);
	}
	return 18u + xz_tree<LCLP>(P, S, base + XZ_LEN_HIGH - 1u, 8, range, code, ip, iend, in);
}

// Input offset of the LZMA2 data of the next block that has chunks, behind the end byte of a block at p - 1: hops block
// padding, the check field, blocks without chunks and, between streams, the index, the footer, stream padding and the next
// stream header (all validated by the walk).  Updates the check size and the dictionary size.  Every read is bounded by the
// payload's n bytes; running past them returns n (which the caller rejects: the walk said more output follows).
__device__ __forceinline__ uint32_t xz_hop(const uint8_t *in, uint32_t n, uint32_t p, uint32_t &csize, uint32_t &dict) {
	auto at = [&](uint32_t x) { return x < n ? (uint32_t)in[x] : 0u; };
	p = ((p + 3u) & ~3u) + csize;   // every structure of a payload starts 4-aligned
	while (p < n) {
		const uint32_t b0 = at(p);
		if (b0) {
			const uint32_t bf = at(p + 1);
			uint32_t x = p + 2;
			for (uint32_t v = 0; v < ((bf >> 6) & 1u) + (bf >> 7) + 2u; v++) {   // the size fields, the filter ID, the property size
				while (at(x++) & 0x80u) {
				}
			}
			dict = xz_dict_size(min(at(x), 40u));
			const uint32_t data = p + (b0 + 1u) * 4u;
			if (at(data) != 0) {
				return data;
			}
			p = ((data + 1u + 3u) & ~3u) + csize;   // a block without chunks
			continue;
		}
		const uint32_t istart = p++;
		uint64_t cnt = 0;
		for (uint32_t sh = 0; sh < 63; sh += 7) {
			const uint32_t b = at(p++);
			cnt |= (uint64_t)(b & 0x7Fu) << sh;
			if (!(b & 0x80u)) {
				break;
			}
		}
		for (uint64_t i = 0; i < 2 * cnt && p < n; i++) {
			while (at(p++) & 0x80u) {
			}
		}
		p = istart + ((p - istart + 3u) & ~3u) + 4u + 12u;
		while (p < n && in[p] == 0) {
			p++;   // stream padding; a later segment means another stream follows
		}
		csize = xz_check_bytes(at(p + 7) & 15u);
		p += 12;
	}
	return n;
}

template <int LCLP>
__global__ void __launch_bounds__(32) k_lzma(const uint8_t *__restrict__ archive, uint8_t *__restrict__ out, const otz_entry *__restrict__ ents,
	const OtzEntryState *__restrict__ est, const uint32_t *__restrict__ list, XzEnt *__restrict__ xe, XzSeg *__restrict__ segs,
	uint32_t n_slots, uint32_t *__restrict__ counter, const uint32_t *__restrict__ n_class) {
	extern __shared__ __align__(16) uint8_t smem_raw[];
	XzSmem<LCLP> &S = *reinterpret_cast<XzSmem<LCLP> *>(smem_raw);
	uint16_t *const P = S.probs;
	auto tile = cg::tiled_partition<32>(cg::this_thread_block());
	const int lane = tile.thread_rank();
	constexpr uint32_t MASK = XZ_RING - 1u;
	constexpr uint32_t SEG = OutRing<32, XZ_RING>::SEG;
	if (*n_class == 0) {
		return;   // no segment of this class in the run
	}
	for (;;) {
		uint32_t s = 0;
		if (lane == 0) {
			s = atomicAdd(counter, 1u);
		}
		s = tile.shfl(s, 0);
		if (s >= n_slots) {
			break;
		}
		const XzSeg sg = segs[s];
		if (sg.k == XZ_NO_SEG || ((sg.meta & 0xFFu) > 3u) != (LCLP == 4)) {
			continue;   // empty slot, or a segment of the other shared-memory class
		}
		const uint32_t ei = list[sg.k];
		const otz_entry e = ents[ei];
		const uint8_t *in = archive + est[ei].data_ofs;
		uint8_t *dst = out + e.out_ofs + sg.out_ofs;
		OutRing<32, XZ_RING> ring;
		ring.init(S.ring, dst);
		const uint32_t q_end = ring.q + sg.out_bytes;
		const uint32_t n = e.comp_size;
		// lane 0's decoder state
		uint32_t q = ring.q, base = ring.q, hp = sg.in_ofs, csize = sg.meta >> 8, dict = sg.dict;
		uint32_t left = 0, lzma_chunk = 0, ip = 0, iend = 0, range = 0, code = 0;
		uint32_t lc = 0, lpm = 0, pbm = 0, st = 0, rep0 = 0, rep1 = 0, rep2 = 0, rep3 = 0;
		int32_t verdict = OTZ_ST_OK;
		for (;;) {
			uint32_t act = XZ_ACT_FLUSH, a0 = 0, a1 = 0;
			tile.sync();
			if (lane == 0) {
				for (;;) {
					if (left == 0) {
						// ---- end of a chunk, start of the next
						if (lzma_chunk) {
							XZ_NORM();
							if (ip != iend || code != 0) {
								act = XZ_ACT_ERR;
								break;
							}
							hp = iend;
							lzma_chunk = 0;
						}
						if (q == q_end) {
							act = XZ_ACT_DONE;
							break;
						}
						// (the walk validated these headers; the bounds below keep a segment inside its payload and its output
						// whatever the bytes say)
						uint32_t c = hp < n ? in[hp] : 0u;
						if (c == 0) {
							hp = xz_hop(in, n, hp + 1u, csize, dict);
							c = hp < n ? in[hp] : 0u;
						}
						if (c == 0 || hp + 6u > n) {
							act = XZ_ACT_ERR;
							break;
						}
						if (c == 1 || c >= 0xE0) {
							base = q;   // dictionary reset
						}
						if (c < 0x80) {
							left = (in[hp + 1] << 8) + in[hp + 2] + 1u;
							if (left > q_end - q || hp + 3u + left > n) {
								act = XZ_ACT_ERR;
								break;
							}
							act = XZ_ACT_RAW;
							a0 = hp + 3u;
							a1 = left;
							hp += 3u + left;
							left = 0;
							break;
						}
						left = ((c & 0x1Fu) << 16) + (in[hp + 1] << 8) + in[hp + 2] + 1u;
						const uint32_t pk = (in[hp + 3] << 8) + in[hp + 4] + 1u;
						ip = hp + 5u;
						if (c >= 0xC0) {
							const uint32_t pr = in[ip++];
							lc = pr % 9u;
							lpm = (1u << (pr / 9u % 5u)) - 1u;
							pbm = (1u << (pr / 45u)) - 1u;
						}
						if (left > q_end - q || ip + pk > n || lc + 31u - __clz(lpm + 1u) > LCLP) {
							act = XZ_ACT_ERR;
							break;
						}
						iend = ip + pk;
						lzma_chunk = 1;
						if (c >= 0xA0) {
							st = rep0 = rep1 = rep2 = rep3 = 0;
						}
						// range decoder init: a zero byte, then the code
						if (pk < 5 || in[ip] != 0) {
							act = XZ_ACT_ERR;
							break;
						}
						code = ((uint32_t)in[ip + 1] << 24) | ((uint32_t)in[ip + 2] << 16) | ((uint32_t)in[ip + 3] << 8) | in[ip + 4];
						range = 0xFFFFFFFFu;
						ip += 5;
						if (c >= 0xA0) {
							act = XZ_ACT_INIT;
							a0 = XZ_P_LIT + (0x300u << (lc + 31u - __clz(lpm + 1u)));
							break;
						}
					}
					if (q - ring.qf >= SEG) {
						break;   // XZ_ACT_FLUSH
					}
					// ---- one LZMA symbol
					const uint32_t pos = q - base, ps = pos & pbm;
					uint32_t b;
					XZ_BIT(XZ_P_ISMATCH + st * 16u + ps, b);
					if (!b) {
						const uint32_t prev = pos ? S.ring[(q - 1u) & MASK] : 0u;
						const uint32_t li = XZ_P_LIT + 0x300u * (((pos & lpm) << lc) + (prev >> (8u - lc)));
						uint32_t m = 1;
						if (st >= 7) {
							uint32_t mb = rep0 < XZ_RING ? S.ring[(q - rep0 - 1u) & MASK] : ring.gbase[q - rep0 - 1u];
							do {
								const uint32_t mbit = (mb >> 7) & 1u;
								mb <<= 1;
								XZ_BIT(li + 0x100u + (mbit << 8) + m, b);
								m = (m << 1) | b;
								if (b != mbit) {
									break;
								}
							} while (m < 0x100u);
						}
						while (m < 0x100u) {
							XZ_BIT(li + m, b);
							m = (m << 1) | b;
						}
						OTZ_CHK(q < q_end, OTZ_CK_XZ_OUT);
						S.ring[q & MASK] = (uint8_t)m;
						q++;
						left--;
						st = st < 4 ? 0 : st < 10 ? st - 3 : st - 6;
						continue;
					}
					uint32_t len;
					XZ_BIT(XZ_P_ISREP + st, b);
					if (!b) {
						len = xz_len<LCLP>(P, S, XZ_P_LEN, ps, range, code, ip, iend, in);
						const uint32_t slot = xz_tree<LCLP>(P, S, XZ_P_SLOT + min(len - 2u, 3u) * 64u - 1u, 6, range, code, ip, iend, in);
						uint32_t dist = slot;
						if (slot >= 4) {
							const int nd = (int)(slot >> 1) - 1;
							dist = (2u | (slot & 1u)) << nd;
							if (slot < 14) {
								dist += xz_rtree<LCLP>(P, S, XZ_P_SPEC + dist - slot - 1u, nd, range, code, ip, iend, in);
							} else {
								uint32_t v = 0;
								for (int i = 0; i < nd - 4; i++) {
									XZ_NORM();
									range >>= 1;
									const uint32_t t = code >= range;
									code -= t ? range : 0u;
									v = (v << 1) | t;
								}
								dist += v << 4;
								dist += xz_rtree<LCLP>(P, S, XZ_P_ALIGN - 1u, 4, range, code, ip, iend, in);
								if (dist == 0xFFFFFFFFu) {
									act = XZ_ACT_ERR;   // end-of-stream marker: not allowed in LZMA2
									break;
								}
							}
						}
						rep3 = rep2;
						rep2 = rep1;
						rep1 = rep0;
						rep0 = dist;
						st = st < 7 ? 7 : 10;
					} else {
						XZ_BIT(XZ_P_ISREP0 + st, b);
						if (!b) {
							XZ_BIT(XZ_P_ISREP0L + st * 16u + ps, b);
							if (!b) {
								// short rep: one byte at rep0
								if (rep0 >= pos || rep0 >= dict) {
									act = XZ_ACT_ERR;
									break;
								}
								st = st < 7 ? 9 : 11;
								OTZ_CHK(q < q_end, OTZ_CK_XZ_OUT);
								S.ring[q & MASK] = rep0 < XZ_RING ? S.ring[(q - rep0 - 1u) & MASK] : ring.gbase[q - rep0 - 1u];
								q++;
								left--;
								continue;
							}
						} else {
							uint32_t d;
							XZ_BIT(XZ_P_ISREP1 + st, b);
							if (!b) {
								d = rep1;
							} else {
								XZ_BIT(XZ_P_ISREP2 + st, b);
								if (!b) {
									d = rep2;
								} else {
									d = rep3;
									rep3 = rep2;
								}
								rep2 = rep1;
							}
							rep1 = rep0;
							rep0 = d;
						}
						len = xz_len<LCLP>(P, S, XZ_P_REPLEN, ps, range, code, ip, iend, in);
						st = st < 7 ? 8 : 11;
					}
					if (rep0 >= pos || rep0 >= dict || len > left) {
						act = XZ_ACT_ERR;   // before the last reset / beyond the dictionary / across the end of the chunk
						break;
					}
					left -= len;
					if (len <= XZ_LANE0_MAX && rep0 < XZ_RING) {
						OTZ_CHK(q + len <= q_end, OTZ_CK_XZ_OUT);
						for (uint32_t i = 0; i < len; i++) {
							S.ring[(q + i) & MASK] = S.ring[(q + i - rep0 - 1u) & MASK];
						}
						q += len;
						continue;
					}
					act = XZ_ACT_COPY;
					a0 = rep0 + 1u;
					a1 = len;
					break;
				}
			}
			act = tile.shfl(act, 0);
			a0 = tile.shfl(a0, 0);
			a1 = tile.shfl(a1, 0);
			ring.q = tile.shfl(q, 0);
			if (act == XZ_ACT_DONE || act == XZ_ACT_ERR) {
				verdict = act == XZ_ACT_ERR ? OTZ_ST_DATA : OTZ_ST_OK;
				break;
			}
			if (act == XZ_ACT_INIT) {
				for (uint32_t i = lane; i < a0; i += 32) {
					P[i] = 1024;
				}
			} else if (act == XZ_ACT_COPY) {
				OTZ_CHK(ring.q + a1 <= q_end, OTZ_CK_XZ_OUT);
				inf_copy<32, XZ_RING>(tile, ring, S.ring, ring.q, a0, a1, lane);
				ring.q += a1;
				q = ring.q;
			} else if (act == XZ_ACT_RAW) {
				OTZ_CHK(ring.q + a1 <= q_end, OTZ_CK_XZ_OUT);
				for (uint32_t done = 0; done < a1;) {
					const uint32_t k = min(a1 - done, SEG);
					for (uint32_t i = lane; i < k; i += 32) {
						OTZ_CHK(a0 + done + i < n, OTZ_CK_XZ_IN);
						S.ring[(ring.q + i) & MASK] = in[a0 + done + i];
					}
					ring.q += k;
					done += k;
					ring.maybe_flush(tile, lane);
				}
				q = ring.q;
			}
			ring.maybe_flush(tile, lane);
		}
		if (verdict == OTZ_ST_OK) {
			ring.finish(tile, lane);
		} else if (lane == 0) {
			// stream order = slot order; the slot is this warp's alone, so it keeps the bytes made before the error for produced[]
			segs[s].made = ring.q - (q_end - sg.out_bytes);
			atomicMin(&xe[sg.k].err, ((unsigned long long)s << 8) | (unsigned)verdict);
		}
	}
}

// Verdict and produced bytes of every XZ entry, and the zero tail of a short one; one warp per entry.
__global__ void __launch_bounds__(256) k_xz_finish(uint8_t *__restrict__ out, const otz_entry *__restrict__ ents, int32_t *__restrict__ status,
	uint32_t *__restrict__ produced, const uint32_t *__restrict__ list, uint32_t n_list, const XzEnt *__restrict__ xe,
	const XzSeg *__restrict__ segs) {
	const uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) / 32u;
	const uint32_t lane = threadIdx.x & 31u;
	if (k >= n_list) {
		return;
	}
	const uint32_t ei = list[k];
	const XzEnt x = xe[k];
	const otz_entry e = ents[ei];
	int32_t st = x.walk_st;
	uint32_t made = x.walk_out;   // every walked chunk decoded
	if (x.err != ~0ull) {
		// the first failing segment precedes the walk's error, which ends the last segment; the segments before it decoded
		st = (int32_t)(x.err & 0xFFu);
		const XzSeg f = segs[x.err >> 8];
		made = f.out_ofs + f.made;
	}
	if (st == OTZ_ST_OK) {
		st = OTZ_ST_OK | OTZ_STF_REF_EOB | (x.walk_out < e.uncomp_size ? OTZ_STF_SHORT : 0);   // the reference rejects method 95
		for (uint64_t i = (uint64_t)x.walk_out + lane; i < e.uncomp_size; i += 32) {
			out[e.out_ofs + i] = 0;
		}
	}
	if (lane == 0) {
		status[ei] = st;
		produced[ei] = made;
	}
}

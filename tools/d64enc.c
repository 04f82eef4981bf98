/* d64enc.c — a small Deflate64 / DEFLATE encoder for the tests and the Deflate64 benchmark (tests/deflate64.py loads it
 * with ctypes as tools/libd64enc.so; `make tools/libd64enc.so`).  Not part of the library: the library reads Deflate64
 * and never writes it.
 *
 *   mode 0  deflate64  64 KiB window, matches up to 65,538 bytes (length symbol 285 = 3 + 16 extra bits, distance
 *                      symbols 30 / 31)
 *   mode 1  dual       32 KiB window, matches up to 257 bytes: the stream is valid DEFLATE and valid Deflate64 with the
 *                      same meaning (the two formats differ only in symbol 285 and distance symbols 30 / 31)
 *   mode 2  deflate    RFC 1951
 *   block 0 dynamic, 1 fixed, 2 stored, 3 cycle through the three
 *
 * Greedy hash-chain LZ77 (`chain` candidates per position), blocks of up to 16,384 symbols, length-limited Huffman codes
 * (the count adjustment of miniz's tdefl_huffman_enforce_max_code_size).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define HBITS 15
#define BLOCK_SYMS 16384

typedef struct {
	uint8_t *out;
	uint64_t cap, n;
	uint64_t acc;
	int nb;
	int overflow;
} Bw;

static void put(Bw *b, uint32_t v, int n) {
	b->acc |= (uint64_t)v << b->nb;
	b->nb += n;
	while (b->nb >= 8) {
		if (b->n < b->cap) {
			b->out[b->n] = (uint8_t)b->acc;
		} else {
			b->overflow = 1;
		}
		b->n++;
		b->acc >>= 8;
		b->nb -= 8;
	}
}
static void align(Bw *b) {
	if (b->nb) {
		put(b, 0, 8 - b->nb);
	}
}

static const uint16_t LBASE[29] = { 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258 };
static const uint8_t LXB[29] = { 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0 };
static const uint32_t DBASE[32] = { 1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
	4097, 6145, 8193, 12289, 16385, 24577, 32769, 49153 };
static const uint8_t DXB[32] = { 0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13, 14, 14 };
static const uint8_t CL_ORDER[19] = { 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15 };

/* symbol of a match length: (symbol - 257, extra bits, extra value) */
static void len_code(uint32_t len, int d64, int *code, int *xb, uint32_t *xv) {
	if (d64 && len >= 258) {
		*code = 28, *xb = 16, *xv = len - 3;
		return;
	}
	if (!d64 && len == 258) {
		*code = 28, *xb = 0, *xv = 0;
		return;
	}
	int c = 27;
	while (LBASE[c] > len) {
		c--;
	}
	*code = c, *xb = LXB[c], *xv = len - LBASE[c];
}
static void dist_code(uint32_t d, int *code, int *xb, uint32_t *xv) {
	int c = 31;
	while (DBASE[c] > d) {
		c--;
	}
	*code = c, *xb = DXB[c], *xv = d - DBASE[c];
}

/* Huffman code lengths (<= maxlen) for n symbols of frequency f; at least two symbols get a code */
static void huff_lengths(const uint32_t *f, int n, int maxlen, uint8_t *len) {
	int sym[320], cnt = 0;
	uint64_t w[640];
	int parent[640];
	memset(len, 0, n);
	for (int i = 0; i < n; i++) {
		if (f[i]) {
			sym[cnt++] = i;
		}
	}
	if (cnt == 0) {
		return;
	}
	if (cnt == 1) {
		len[sym[0]] = 1;
		return;
	}
	/* sort symbols by frequency (insertion sort: n <= 288) */
	for (int i = 1; i < cnt; i++) {
		int s = sym[i], j = i - 1;
		while (j >= 0 && f[sym[j]] > f[s]) {
			sym[j + 1] = sym[j];
			j--;
		}
		sym[j + 1] = s;
	}
	/* two-queue Huffman: leaves 0..cnt-1 (sorted), internal nodes cnt.. in creation order */
	for (int i = 0; i < cnt; i++) {
		w[i] = f[sym[i]];
	}
	int li = 0, ii = cnt, nn = cnt;
	for (int k = 0; k < cnt - 1; k++) {
		int pick[2];
		for (int t = 0; t < 2; t++) {
			if (li < cnt && (ii >= nn || w[li] <= w[ii])) {
				pick[t] = li++;
			} else {
				pick[t] = ii++;
			}
		}
		w[nn] = w[pick[0]] + w[pick[1]];
		parent[pick[0]] = parent[pick[1]] = nn;
		nn++;
	}
	int depth[640];
	depth[nn - 1] = 0;
	for (int i = nn - 2; i >= 0; i--) {
		depth[i] = depth[parent[i]] + 1;
	}
	int num[33] = { 0 };
	for (int i = 0; i < cnt; i++) {
		num[depth[i] > 32 ? 32 : depth[i]]++;
	}
	for (int i = maxlen + 1; i <= 32; i++) {
		num[maxlen] += num[i];
		num[i] = 0;
	}
	uint32_t total = 0;
	for (int i = maxlen; i > 0; i--) {
		total += (uint32_t)num[i] << (maxlen - i);
	}
	while (total != (1u << maxlen)) {
		num[maxlen]--;
		for (int i = maxlen - 1; i > 0; i--) {
			if (num[i]) {
				num[i]--;
				num[i + 1] += 2;
				break;
			}
		}
		total--;
	}
	/* most frequent symbols (end of sym[]) get the shortest codes */
	int k = cnt - 1;
	for (int l = 1; l <= maxlen; l++) {
		for (int c = 0; c < num[l]; c++) {
			len[sym[k--]] = (uint8_t)l;
		}
	}
}

static void canon(const uint8_t *len, int n, uint16_t *code) {
	int cnt[16] = { 0 }, next[16];
	for (int i = 0; i < n; i++) {
		cnt[len[i]]++;
	}
	cnt[0] = 0;
	int c = 0;
	for (int l = 1; l < 16; l++) {
		c = (c + cnt[l - 1]) << 1;
		next[l] = c;
	}
	for (int i = 0; i < n; i++) {
		if (len[i]) {
			uint32_t v = (uint32_t)next[len[i]]++, r = 0;
			for (int b = 0; b < len[i]; b++) {
				r = (r << 1) | ((v >> b) & 1u);
			}
			code[i] = (uint16_t)r;
		}
	}
}

typedef struct {
	uint32_t len, dist;   /* len 0: literal `dist` */
} Tok;

static void emit_block(Bw *b, const Tok *t, int nt, int final, int kind, int d64, const uint8_t *src, uint32_t raw_n) {
	if (kind == 2) {
		/* stored: the raw bytes of these tokens, in pieces of at most 65,535 */
		uint32_t o = 0;
		do {
			uint32_t n = raw_n - o > 65535u ? 65535u : raw_n - o;
			put(b, (final && o + n == raw_n) ? 1u : 0u, 1);
			put(b, 0, 2);
			align(b);
			put(b, n & 0xFFFF, 16);
			put(b, ~n & 0xFFFF, 16);
			for (uint32_t i = 0; i < n; i++) {
				put(b, src[o + i], 8);
			}
			o += n;
		} while (o < raw_n);
		return;
	}
	uint8_t ll[288], dl[32];
	uint16_t lc[288], dc[32];
	int hlit = 286, hdist = d64 ? 32 : 30;
	if (kind == 1) {
		for (int i = 0; i < 288; i++) {
			ll[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
		}
		for (int i = 0; i < 32; i++) {
			dl[i] = 5;
		}
	} else {
		uint32_t lf[288] = { 0 }, df[32] = { 0 };
		for (int i = 0; i < nt; i++) {
			if (!t[i].len) {
				lf[t[i].dist]++;
			} else {
				int c, xb, dcd;
				uint32_t xv;
				len_code(t[i].len, d64, &c, &xb, &xv);
				lf[257 + c]++;
				dist_code(t[i].dist, &dcd, &xb, &xv);
				df[dcd]++;
			}
		}
		lf[256]++;
		int nl = 0;
		for (int i = 0; i < 286; i++) {
			nl += lf[i] != 0;
		}
		if (nl < 2) {
			lf[0]++;   /* at least two codes (as zlib's deflate does) */
		}
		int nd = 0;
		for (int i = 0; i < 32; i++) {
			nd += df[i] != 0;
		}
		if (nd < 2) {
			df[df[0] ? 1 : 0]++;
			if (nd == 0) {
				df[1]++;
			}
		}
		huff_lengths(lf, 286, 15, ll);
		huff_lengths(df, d64 ? 32 : 30, 15, dl);
		while (hlit > 257 && !ll[hlit - 1]) {
			hlit--;
		}
		while (hdist > 1 && !dl[hdist - 1]) {
			hdist--;
		}
	}
	canon(ll, kind == 1 ? 288 : 286, lc);
	canon(dl, kind == 1 ? 32 : (d64 ? 32 : 30), dc);
	put(b, final ? 1u : 0u, 1);
	put(b, kind == 1 ? 1u : 2u, 2);
	if (kind == 0) {
		/* code lengths, run-length coded with 16 / 17 / 18 */
		uint8_t all[320];
		int na = 0;
		memcpy(all, ll, hlit);
		memcpy(all + hlit, dl, hdist);
		na = hlit + hdist;
		uint16_t rs[320], rx[320];
		int nr = 0;
		for (int i = 0; i < na;) {
			int r = 1;
			while (i + r < na && all[i + r] == all[i]) {
				r++;
			}
			if (all[i] == 0 && r >= 3) {
				int n = r > 138 ? 138 : r;
				if (n >= 11) {
					rs[nr] = 18, rx[nr++] = (uint16_t)(n - 11);
				} else {
					rs[nr] = 17, rx[nr++] = (uint16_t)(n - 3);
				}
				i += n;
			} else if (all[i] != 0 && r >= 4) {
				rs[nr] = all[i], rx[nr++] = 0;
				int n = r - 1 > 6 ? 6 : r - 1;
				rs[nr] = 16, rx[nr++] = (uint16_t)(n - 3);
				i += 1 + n;
			} else {
				rs[nr] = all[i], rx[nr++] = 0;
				i++;
			}
		}
		uint32_t cf[19] = { 0 };
		for (int i = 0; i < nr; i++) {
			cf[rs[i]]++;
		}
		int ncf = 0;
		for (int i = 0; i < 19; i++) {
			ncf += cf[i] != 0;
		}
		if (ncf < 2) {
			cf[cf[0] ? 1 : 0]++;   /* the code-length code must be complete: two codes at least */
		}
		uint8_t cl[19];
		uint16_t cc[19];
		huff_lengths(cf, 19, 7, cl);
		canon(cl, 19, cc);
		int hclen = 19;
		while (hclen > 4 && !cl[CL_ORDER[hclen - 1]]) {
			hclen--;
		}
		put(b, (uint32_t)(hlit - 257), 5);
		put(b, (uint32_t)(hdist - 1), 5);
		put(b, (uint32_t)(hclen - 4), 4);
		for (int i = 0; i < hclen; i++) {
			put(b, cl[CL_ORDER[i]], 3);
		}
		for (int i = 0; i < nr; i++) {
			put(b, cc[rs[i]], cl[rs[i]]);
			if (rs[i] == 16) {
				put(b, rx[i], 2);
			} else if (rs[i] == 17) {
				put(b, rx[i], 3);
			} else if (rs[i] == 18) {
				put(b, rx[i], 7);
			}
		}
	}
	for (int i = 0; i < nt; i++) {
		if (!t[i].len) {
			put(b, lc[t[i].dist], ll[t[i].dist]);
			continue;
		}
		int c, xb, dcd;
		uint32_t xv;
		len_code(t[i].len, d64, &c, &xb, &xv);
		put(b, lc[257 + c], ll[257 + c]);
		if (xb) {
			put(b, xv, xb);
		}
		dist_code(t[i].dist, &dcd, &xb, &xv);
		put(b, dc[dcd], dl[dcd]);
		if (xb) {
			put(b, xv, xb);
		}
	}
	put(b, lc[256], ll[256]);
}

uint64_t d64enc_bound(uint64_t n) { return n + (n >> 3) + 5 * (n / 16384 + 1) + 1024; }

/* Returns the stream length, -1 when `cap` is too small, -2 on a bad argument / no memory. */
int64_t d64enc(const uint8_t *in, uint64_t n, uint8_t *out, uint64_t cap, int mode, int block, int chain) {
	if (mode < 0 || mode > 2 || block < 0 || block > 3) {
		return -2;
	}
	const int d64 = mode == 0;
	const uint32_t win = d64 ? 65536u : 32768u;
	const uint32_t maxm = mode == 0 ? 65538u : mode == 1 ? 257u : 258u;
	int32_t *head = (int32_t *)malloc(sizeof(int32_t) << HBITS);
	int32_t *prev = (int32_t *)malloc(sizeof(int32_t) * (size_t)win);
	Tok *tok = (Tok *)malloc(sizeof(Tok) * BLOCK_SYMS);
	if (!head || !prev || !tok) {
		free(head), free(prev), free(tok);
		return -2;
	}
	for (uint32_t i = 0; i < (1u << HBITS); i++) {
		head[i] = -1;
	}
	Bw b = { out, cap, 0, 0, 0, 0 };
	uint64_t p = 0, blk_start = 0;
	int nt = 0, kind = block == 3 ? 0 : block;
#define HASH(q) ((((uint32_t)in[q] << 10) ^ ((uint32_t)in[(q) + 1] << 5) ^ in[(q) + 2]) & ((1u << HBITS) - 1u))
#define INSERT(q)                                 \
	do {                                          \
		if ((q) + 2 < n) {                        \
			uint32_t h_ = HASH(q);                \
			prev[(q) & (win - 1)] = head[h_];     \
			head[h_] = (int32_t)(q);              \
		}                                         \
	} while (0)
	if (n == 0) {
		emit_block(&b, NULL, 0, 1, kind == 2 ? 0 : kind, d64, in, 0);
	}
	while (p < n) {
		uint32_t best = 0, bd = 0;
		if (p + 2 < n) {
			int32_t c = head[HASH(p)];
			int left = chain;
			const uint64_t lim = n - p < maxm ? n - p : maxm;
			while (c >= 0 && left-- > 0 && p - (uint64_t)c <= win) {
				const uint8_t *a = in + p, *s = in + c;
				if (s[best] == a[best] || best == 0) {
					uint32_t l = 0;
					while (l < lim && a[l] == s[l]) {
						l++;
					}
					if (l > best) {
						best = l, bd = (uint32_t)(p - (uint64_t)c);
						if (l == lim) {
							break;
						}
					}
				}
				int32_t nx = prev[c & (win - 1)];
				if (nx >= c) {
					break;
				}
				c = nx;
			}
		}
		if (best >= 3) {
			tok[nt].len = best, tok[nt].dist = bd;
			for (uint32_t i = 0; i < best; i++) {
				INSERT(p + i);
			}
			p += best;
		} else {
			tok[nt].len = 0, tok[nt].dist = in[p];
			INSERT(p);
			p++;
		}
		nt++;
		if (nt == BLOCK_SYMS || p == n) {
			emit_block(&b, tok, nt, p == n, kind, d64, in + blk_start, (uint32_t)(p - blk_start));
			blk_start = p;
			nt = 0;
			if (block == 3) {
				kind = (kind + 1) % 3;
			}
		}
	}
	align(&b);
	free(head), free(prev), free(tok);
	return b.overflow ? -1 : (int64_t)b.n;
}

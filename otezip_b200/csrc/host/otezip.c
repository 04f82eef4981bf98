/* otezip.c — plain-C99 host side of the B200 build: the libzip-subset API of include/otezip/zip.h
 * over the batched GPU codec behind include/otz_gpu.h.
 *
 * Mirrors the reference's container layer and API (paths relative to /root/reference):
 *   EOCD search + central-directory walk     src/lib/otezip.c:199-396   (same accept/reject rules; the
 *                                             walk now also emits the device entry table)
 *   zip_open / zip_close / accessors         src/lib/otezip.c:693-785, :1273-1404
 *   zip_fopen_index / zip_fclose / zip_fread src/lib/otezip.c:1315-1357 (+ otezip_extract_entry :399-684)
 *   zip_file_add / zip_set_file_compression  src/lib/otezip.c:1079-1237
 *   LFH / CDH / EOCD writers                 src/lib/otezip.c:1443-1590 (exact field values)
 *   DOS time                                 src/lib/time.inc.c:29-70
 * There is no codec in this file and no CPU fallback: every decode, encode and CRC goes through
 * otz_extract_host() / otz_deflate_host().  Without a CUDA device zip_fopen_index() returns NULL and
 * zip_close() of a written archive returns -1, each with a message on stderr.
 */
#include <errno.h>
#include <fcntl.h>
#include <sys/random.h>
#include <sys/stat.h>
#include <unistd.h>

#include "otezip/zip.h"
#include "otz_gpu.h"

#define SIG_LFH 0x04034b50u
#define SIG_CDH 0x02014b50u
#define SIG_EOCD 0x06054b50u
#define MAX_FIELD_LEN 65535u                            /* otezip.c:101 */
#define MAX_PAYLOAD (2ULL * 1024 * 1024 * 1024)         /* otezip.c:102 */
#define ERR_READ (-1)                                   /* otezip.c:191 */
#define ERR_INCONS (-2)                                 /* otezip.c:192 */
/* Chunk index: LFH extra field written for multi-chunk DEFLATE entries (ignored by the reference, which skips
 * extra fields, otezip.c:429-437): id 'OZ', then {u8 version=1, u8 0, u16 0, u32 chunk_bytes, u32 n_chunks,
 * u32 csize[n_chunks]}.  Each chunk is an independently decodable run of DEFLATE blocks (k_deflate.cuh). */
#define OZ_EXTRA_ID 0x5A4Fu
#define OZ_EXTRA_MAX_CHUNKS 16000u
/* WinZip AES (AE-1 / AE-2): method 99, flag bit 0, extra field 0x9901 = {u16 vendor version 1|2, 'A' 'E', u8 strength 1-3,
 * u16 actual method}; payload = salt (8/12/16) | verification value (2) | ciphertext | authentication code (10) */
#define METHOD_AES 99u
#define AES_EXTRA_ID 0x9901u
#define AES_OVERHEAD(strength) (4u + 4u * (strength) + 2u + 10u)

/* otezip.c:157-166 */
int otezip_verify_crc = 0;
uint64_t otezip_max_expansion_ratio = 1000ULL;
uint64_t otezip_max_expansion_slack = 1024ULL * 1024ULL;
int otezip_ignore_zipbomb = 0;
int otezip_ref_compat = 1;
int otezip_write_data_descriptors = 0;
int otezip_zstd_frames = 0;

/* OTEZIP_REF_COMPAT=0 in the environment sets the initial value of otezip_ref_compat, so that a program that never touches
 * the global (the otezip CLI) can extract what the reference rejects: Deflate64 and XZ entries, F1 streams, real Zstandard frames.
 * Read once, when the library is loaded; a program that assigns the global later still wins. */
__attribute__ ((constructor)) static void otezip_env_defaults(void) {
	const char *e = getenv ("OTEZIP_REF_COMPAT");
	if (e && *e) {
		otezip_ref_compat = atoi (e) != 0;
	}
}

/* ---- private archive state; `pub` must stay first: zip_t* == struct otz_archive* ---- */
struct otz_window {               /* one decoded batch of consecutive entries */
	struct otz_window *next;
	zip_uint64_t first, last;     /* entries [first, last) */
	uint8_t *arena;               /* pinned host memory holding the decoded bytes */
	uint64_t arena_len;
	uint64_t *ofs;                /* per entry offset into arena */
	int32_t *status;
	uint32_t *crc;
	uint32_t refs;                /* zip_file_t handles pointing into arena */
	int current;
	int orphan;                   /* its archive was closed while handles were still open: the last zip_fclose frees it */
	uint32_t pw_gen;              /* default password its AES entries were decoded with (otz_archive.pw_gen) */
};

struct otz_pending {              /* a queued source (write path) */
	void *buf;
	uint64_t len;
	int owned;                    /* free(buf) after the archive is written */
	int dirty;                    /* has bytes that zip_close must write (every new entry; a replaced existing one) */
	uint32_t level;               /* compression level asked for with zip_set_file_compression (libzip: 0 = default, 1-9) */
	uint16_t enc;                 /* zip_file_set_encryption: AES strength 1-3, 0 = none */
	char *pw;                     /* its password; NULL = the default password at zip_close */
};

struct otz_aesx {                 /* the 0x9901 field of an entry whose directory method is 99 */
	uint16_t vendor;              /* 1 = AE-1, 2 = AE-2; 0 = no usable field (the entry is rejected with OTZ_ST_METHOD) */
	uint8_t strength;
	uint16_t method;              /* actual compression method */
};

static int index_enabled(void) {
	const char *e = getenv ("OTEZIP_NO_INDEX");
	return !(e && e[0] == '1');
}

struct otz_archive {
	struct zip pub;
	uint32_t magic;
	char *path;
	/* read side */
	uint8_t *image;               /* pinned copy of the archive file (filled on first extract) */
	uint64_t image_len;
	struct otz_window *windows;
	int32_t *last_status;
	uint64_t *lfh64;              /* local header offset of every entry (ZIP64: may exceed the public u32 field) */
	uint64_t lfh64_cap;
	/* write side */
	struct otz_pending *pend;     /* parallel to pub.entries for entries added in this session */
	zip_uint64_t n_existing;      /* entries loaded from an existing archive (append mode) */
	uint64_t append_ofs;          /* where new data starts in append mode */
	/* encryption */
	struct otz_aesx *aes;         /* per entry; vendor 0 for entries that are not AES-encrypted */
	uint64_t aes_cap;
	char *default_pw;
	uint32_t pw_gen;              /* bumped by every zip_set_default_password */
};
#define OTZ_MAGIC 0x5a32424fu

struct otz_file {                 /* zip_file_t plus the window it borrows from */
	struct zip_file pub;
	struct otz_window *win;
	uint8_t *own;                 /* malloc'd data (zero-length entries) */
};

/* Devices of the read path: OTEZIP_DEVICES = "all" or a comma list ("0,2,3") shards every batch of entries over those
 * GPUs (otz_extract_host_multi: contiguous index ranges balanced by bytes, no collective — SURVEY.md §8e); otherwise the
 * one device OTEZIP_DEVICE names (default 0).  The write path and the zlib-compatible single-stream calls use the first. */
#define OTZ_MAX_DEVICES 16
static otz_ctx *g_ctxs[OTZ_MAX_DEVICES];
static uint32_t g_nctx;
static int g_ctx_failed;

static uint32_t otezip_b200_ctxs(otz_ctx ***out) {
	if (!g_nctx && !g_ctx_failed) {
		int devs[OTZ_MAX_DEVICES], nd = 0;
		const char *e = getenv ("OTEZIP_DEVICES");
		if (e && !strcmp (e, "all")) {
			const int have = otz_device_count ();
			for (int d = 0; d < have && nd < OTZ_MAX_DEVICES; d++) {
				devs[nd++] = d;
			}
		} else if (e && *e) {
			const char *q = e;
			while (*q && nd < OTZ_MAX_DEVICES) {
				char *end = NULL;
				long d = strtol (q, &end, 10);
				if (end == q) {
					break;
				}
				devs[nd++] = (int)d;
				q = *end == ',' ? end + 1 : end;
			}
		}
		if (!nd) {
			const char *one = getenv ("OTEZIP_DEVICE");
			devs[nd++] = one ? atoi (one) : 0;
		}
		for (int i = 0; i < nd; i++) {
			if (otz_ctx_create (devs[i], &g_ctxs[g_nctx]) != OTZ_SUCCESS) {
				fprintf (stderr, "otezip-b200: no usable CUDA device %d (%s); this build has no CPU codec\n", devs[i], otz_last_error ());
				for (uint32_t k = 0; k < g_nctx; k++) {
					otz_ctx_destroy (g_ctxs[k]);
					g_ctxs[k] = NULL;
				}
				g_nctx = 0;
				g_ctx_failed = 1;
				break;
			}
			g_nctx++;
		}
	}
	*out = g_ctxs;
	return g_nctx;
}

otz_ctx *otezip_b200_ctx(void);   /* shared with zcompat.c */
otz_ctx *otezip_b200_ctx(void) {
	otz_ctx **c;
	return otezip_b200_ctxs (&c) ? c[0] : NULL;
}

static struct otz_archive *priv(zip_t *za) {
	struct otz_archive *a = (struct otz_archive *)za;
	return (a && a->magic == OTZ_MAGIC) ? a : NULL;
}

static int is_valid(const zip_t *za) {
	return za != NULL && za->fp != NULL; /* otezip.c:687-689 */
}

/* the AES field of entry i, or NULL when its directory method is not 99 (vendor 0: method 99 without a usable field) */
static const struct otz_aesx *aes_of(const struct otz_archive *a, zip_uint64_t i) {
	if (i >= a->pub.n_entries || a->pub.entries[i].method != METHOD_AES) {
		return NULL;
	}
	static const struct otz_aesx none = { 0, 0, 0 };
	return (a->aes && i < a->aes_cap) ? &a->aes[i] : &none;
}

/* compressed bytes the decoder sees: for an AES entry the ciphertext, without salt, verification value and code */
static uint64_t inner_comp(const struct otz_archive *a, zip_uint64_t i) {
	const struct otz_aesx *x = aes_of (a, i);
	const uint64_t c = a->pub.entries[i].comp_size;
	return (x && x->vendor && c >= AES_OVERHEAD (x->strength)) ? c - AES_OVERHEAD (x->strength) : c;
}

static void wipe_free(char *p) {
	if (p) {
		volatile char *v = p;
		while (*v) {
			*v++ = 0;
		}
		free (p);
	}
}

#define OTZ_MAX_ENTRIES (1ull << 24)   /* ZIP64 lifts the 65,535 of the EOCD; this bounds the entry table */

/* local header offset of entry i: 64-bit (the public struct otezip_entry keeps the reference's u32 field) */
static uint64_t entry_lfh(const zip_t *za, zip_uint64_t i) {
	const struct otz_archive *a = (const struct otz_archive *)za;
	return (a->magic == OTZ_MAGIC && a->lfh64 && i < a->lfh64_cap) ? a->lfh64[i] : za->entries[i].local_hdr_ofs;
}

/* ---- method names, otezip.c:112-154 (only what this build implements) ---- */
int otezip_method_from_string(const char *s) {
	if (!s) {
		return -1;
	}
	if (!strcmp (s, "store")) {
		return OTEZIP_METHOD_STORE;
	}
	if (!strcmp (s, "deflate")) {
		return OTEZIP_METHOD_DEFLATE;
	}
	if (!strcmp (s, "zstd")) {
		return OTEZIP_METHOD_ZSTD;
	}
	return -1;
}

/* ---- DOS time, time.inc.c:29-70 ---- */
static int clampi(int v, int lo, int hi) {
	return v < lo ? lo : v > hi ? hi : v;
}
static void dos_now(uint16_t *t, uint16_t *d) {
	time_t now = time (NULL);
	struct tm tmv;
	if (now == (time_t)-1 || !localtime_r (&now, &tmv)) {
		*t = 0;
		*d = (uint16_t)((1 << 5) | 1);
		return;
	}
	*t = (uint16_t)((clampi (tmv.tm_hour, 0, 23) << 11) | (clampi (tmv.tm_min, 0, 59) << 5) | clampi (tmv.tm_sec / 2, 0, 29));
	*d = (uint16_t)((clampi (tmv.tm_year + 1900 - 1980, 0, 127) << 9) | (clampi (tmv.tm_mon + 1, 1, 12) << 5) |
		clampi (tmv.tm_mday, 1, 31));
}

/* ---------------------------------------------------------------- central directory */

static int read_at(FILE *fp, long ofs, void *dst, size_t n) {
	if (fseek (fp, ofs, SEEK_SET) != 0) {
		return -1;
	}
	return fread (dst, 1, n, fp) == n ? 0 : -1;
}

/* otezip.c:199-272: newest EOCD whose directory range lies in the file and starts with a CDH.
 * Beyond the reference (SURVEY.md F5 / §8f rank 2): when the EOCD carries the ZIP64 escape values (0xFFFF entries,
 * 0xFFFFFFFF size or offset) the ZIP64 locator in front of it and the ZIP64 end-of-central-directory record it points
 * to (APPNOTE 4.3.14-4.3.15) supply the 64-bit count, size and offset. */
#define SIG_EOCD64 0x06064b50u
#define SIG_EOCD64_LOC 0x07064b50u
static int find_eocd(FILE *fp, long file_size, uint64_t *cd_size, uint64_t *cd_ofs, uint64_t *n_entries) {
	if (file_size < 22) {
		return ERR_INCONS;
	}
	size_t span = file_size < 0x10000 + 22 ? (size_t)file_size : (size_t)(0x10000 + 22);
	uint8_t *tail = (uint8_t *)malloc (span);
	if (!tail) {
		return ERR_READ;
	}
	if (read_at (fp, file_size - (long)span, tail, span) != 0) {
		free (tail);
		return ERR_READ;
	}
	int rc = ERR_INCONS;
	for (size_t i = span - 22 + 1; i-- > 0;) {
		if (otezip_read_le32 (tail + i) != SIG_EOCD) {
			continue;
		}
		uint64_t ents = otezip_read_le16 (tail + i + 10);
		uint64_t sz = otezip_read_le32 (tail + i + 12), ofs = otezip_read_le32 (tail + i + 16);
		if (ents == 0xFFFFu || sz == 0xFFFFFFFFu || ofs == 0xFFFFFFFFu) {
			const long eocd_pos = file_size - (long)span + (long)i;
			uint8_t loc[20], rec[56];
			if (eocd_pos < 20 || read_at (fp, eocd_pos - 20, loc, 20) != 0 || otezip_read_le32 (loc) != SIG_EOCD64_LOC) {
				continue;
			}
			const uint64_t rpos = (uint64_t)otezip_read_le32 (loc + 8) | ((uint64_t)otezip_read_le32 (loc + 12) << 32);
			if (rpos + 56 > (uint64_t)file_size || read_at (fp, (long)rpos, rec, 56) != 0 || otezip_read_le32 (rec) != SIG_EOCD64) {
				continue;
			}
			ents = (uint64_t)otezip_read_le32 (rec + 32) | ((uint64_t)otezip_read_le32 (rec + 36) << 32);
			sz = (uint64_t)otezip_read_le32 (rec + 40) | ((uint64_t)otezip_read_le32 (rec + 44) << 32);
			ofs = (uint64_t)otezip_read_le32 (rec + 48) | ((uint64_t)otezip_read_le32 (rec + 52) << 32);
		}
		if (ofs > (uint64_t)file_size || sz > (uint64_t)file_size || ofs + sz > (uint64_t)file_size) {
			continue;
		}
		if (ents > 0 && sz >= 4) {
			uint8_t sig[4];
			if (read_at (fp, (long)ofs, sig, 4) != 0 || otezip_read_le32 (sig) != SIG_CDH) {
				continue;
			}
		}
		*n_entries = ents;
		*cd_size = sz;
		*cd_ofs = ofs;
		rc = 0;
		break;
	}
	free (tail);
	return rc;
}

/* otezip.c:275-396 */
static int load_central(struct otz_archive *a) {
	zip_t *za = &a->pub;
	if (fseek (za->fp, 0, SEEK_END) != 0) {
		return ERR_READ;
	}
	long fsz = ftell (za->fp);
	if (fsz < 0) {
		return ERR_READ;
	}
	uint64_t cd_size = 0, cd_ofs = 0, n = 0;
	int rc = find_eocd (za->fp, fsz, &cd_size, &cd_ofs, &n);
	if (rc != 0) {
		return rc;
	}
	if (cd_ofs + cd_size > (uint64_t)fsz || n > OTZ_MAX_ENTRIES) {
		return ERR_INCONS;
	}
	a->append_ofs = cd_ofs;
	if (n == 0) {
		return cd_size != 0 ? ERR_INCONS : 0;
	}
	if ((uint64_t)cd_size > MAX_PAYLOAD) {
		return ERR_INCONS;
	}
	uint8_t *cd = (uint8_t *)malloc (cd_size);
	if (!cd) {
		return ERR_READ;
	}
	if (read_at (za->fp, (long)cd_ofs, cd, cd_size) != 0) {
		free (cd);
		return ERR_READ;
	}
	if ((size_t)n * 46 > cd_size) {
		free (cd);
		return ERR_INCONS;
	}
	za->entries = (struct otezip_entry *)calloc (n, sizeof (struct otezip_entry));
	a->lfh64 = (uint64_t *)calloc (n, sizeof (uint64_t));
	a->lfh64_cap = n;
	a->aes = (struct otz_aesx *)calloc (n, sizeof (struct otz_aesx));
	a->aes_cap = n;
	if (!za->entries || !a->lfh64 || !a->aes) {
		free (cd);
		return ERR_READ;
	}
	za->n_entries = n;
	size_t off = 0;
	for (uint64_t i = 0; i < n; i++) {
		if (off + 46 > cd_size || otezip_read_le32 (cd + off) != SIG_CDH) {
			free (cd);
			return ERR_INCONS;
		}
		const uint8_t *h = cd + off;
		size_t fl = otezip_read_le16 (h + 28), xl = otezip_read_le16 (h + 30), cl = otezip_read_le16 (h + 32);
		if (46 + fl + xl + cl > cd_size - off) {
			free (cd);
			return ERR_INCONS;
		}
		struct otezip_entry *e = &za->entries[i];
		e->method = otezip_read_le16 (h + 10);
		e->file_time = otezip_read_le16 (h + 12);
		e->file_date = otezip_read_le16 (h + 14);
		e->crc32 = otezip_read_le32 (h + 16);
		e->comp_size = otezip_read_le32 (h + 20);
		e->uncomp_size = otezip_read_le32 (h + 24);
		e->external_attr = otezip_read_le32 (h + 38);
		e->local_hdr_ofs = otezip_read_le32 (h + 42);
		uint64_t comp64 = e->comp_size, uncomp64 = e->uncomp_size, lfh = e->local_hdr_ofs;
		const int escaped = e->comp_size == 0xFFFFFFFFu || e->uncomp_size == 0xFFFFFFFFu || e->local_hdr_ofs == 0xFFFFFFFFu;
		if (escaped || e->method == METHOD_AES) {
			/* ZIP64 extended information (APPNOTE 4.5.3): the escaped fields, in this order, 8 bytes each;
			 * WinZip AES field 0x9901 of a method-99 entry */
			const uint8_t *x = h + 46 + fl;
			size_t xo = 0;
			int found = !escaped;
			while (xo + 4 <= xl) {
				const size_t id = otezip_read_le16 (x + xo), sz = otezip_read_le16 (x + xo + 2);
				if (xo + 4 + sz > xl) {
					break;
				}
				if (id == AES_EXTRA_ID && e->method == METHOD_AES) {
					const uint8_t *d = x + xo + 4;
					const uint16_t ver = sz == 7 ? otezip_read_le16 (d) : 0, am = sz == 7 ? otezip_read_le16 (d + 5) : 0xFFFF;
					if ((ver == 1 || ver == 2) && d[2] == 'A' && d[3] == 'E' && d[4] >= 1 && d[4] <= 3 &&
						(am == OTEZIP_METHOD_STORE || am == OTEZIP_METHOD_DEFLATE || am == OTZ_M_DEFLATE64 || am == OTEZIP_METHOD_ZSTD ||
						 am == OTZ_M_XZ)) {
						a->aes[i].vendor = ver;
						a->aes[i].strength = d[4];
						a->aes[i].method = am;
					}
				}
				if (id == 0x0001 && escaped) {
					size_t q = xo + 4;
					const size_t end = xo + 4 + sz;
					found = 1;
					if (e->uncomp_size == 0xFFFFFFFFu) {
						found = found && q + 8 <= end;
						if (found) {
							uncomp64 = (uint64_t)otezip_read_le32 (x + q) | ((uint64_t)otezip_read_le32 (x + q + 4) << 32);
							q += 8;
						}
					}
					if (found && e->comp_size == 0xFFFFFFFFu) {
						found = q + 8 <= end;
						if (found) {
							comp64 = (uint64_t)otezip_read_le32 (x + q) | ((uint64_t)otezip_read_le32 (x + q + 4) << 32);
							q += 8;
						}
					}
					if (found && e->local_hdr_ofs == 0xFFFFFFFFu) {
						found = q + 8 <= end;
						if (found) {
							lfh = (uint64_t)otezip_read_le32 (x + q) | ((uint64_t)otezip_read_le32 (x + q + 4) << 32);
						}
					}
					if (e->method != METHOD_AES) {
						break;
					}
				}
				xo += 4 + sz;
			}
			if (!found) {
				free (cd);
				return ERR_INCONS;
			}
		}
		if (comp64 > MAX_PAYLOAD || uncomp64 > MAX_PAYLOAD) {
			free (cd);
			return ERR_INCONS;
		}
		e->comp_size = (uint32_t)comp64;
		e->uncomp_size = (uint32_t)uncomp64;
		e->local_hdr_ofs = (uint32_t)lfh;   /* public field: low 32 bits; a->lfh64[] is what the library uses */
		a->lfh64[i] = lfh;
		e->name = (char *)malloc (fl + 1);
		if (!e->name) {
			free (cd);
			return ERR_READ;
		}
		memcpy (e->name, h + 46, fl);
		e->name[fl] = '\0';
		off += 46 + fl + xl + cl;
	}
	free (cd);
	return 0;
}

/* The device entry table the walk emits: one otz_entry per directory entry. */
zip_uint64_t otezip_b200_entry_table(zip_t *za, void *rows, zip_uint64_t max_rows) {
	if (!is_valid (za) || !rows) {
		return 0;
	}
	otz_entry *t = (otz_entry *)rows;
	uint64_t out = 0;
	zip_uint64_t n = za->n_entries < max_rows ? za->n_entries : max_rows;
	for (zip_uint64_t i = 0; i < n; i++) {
		const struct otezip_entry *e = &za->entries[i];
		t[i].lfh_ofs = entry_lfh (za, i);
		t[i].out_ofs = out;
		t[i].comp_size = e->comp_size;
		t[i].uncomp_size = e->uncomp_size;
		t[i].crc32 = e->crc32;
		t[i].method = e->method;
		t[i].flags = 0;
		out += ((uint64_t)e->uncomp_size + 15) & ~15ULL;
	}
	return n;
}

/* ---------------------------------------------------------------- open / close */

static void free_windows(struct otz_archive *a);

zip_t *zip_open(const char *path, int flags, int *errorp) {
	struct otz_archive *a = (struct otz_archive *)calloc (1, sizeof (*a));
	if (!a || !path) {
		free (a);
		if (errorp) {
			*errorp = -1;
		}
		return NULL;
	}
	a->magic = OTZ_MAGIC;
	zip_t *za = &a->pub;
	const char *mode = "rb";
	int exists = 0;
	if (flags & ZIP_CREATE) { /* otezip.c:708-738 */
		if ((flags & ZIP_EXCL) && (flags & ZIP_TRUNCATE)) {
			goto fail_flags;
		}
		FILE *probe = fopen (path, "rb");
		exists = probe != NULL;
		if (probe) {
			fclose (probe);
		}
		if (exists && (flags & ZIP_EXCL)) {
			goto fail_flags;
		}
		mode = (exists && !(flags & ZIP_TRUNCATE)) ? "r+b" : "w+b";
		za->mode = 1;
	}
	if (mode[0] == 'w') {
		unlink (path); /* otezip.c:744-747 */
	}
	za->fp = fopen (path, mode);
	if (!za->fp) {
		if (errorp) {
			*errorp = ZIP_ER_OPEN;
		}
		free (a);
		return NULL;
	}
	a->path = strdup (path);
	if (za->mode == 0 || (exists && !(flags & ZIP_TRUNCATE))) { /* otezip.c:758-780 */
		int rc = load_central (a);
		if (rc != 0) {
			if (errorp) {
				*errorp = rc == ERR_READ ? ZIP_ER_READ : rc == ERR_INCONS ? ZIP_ER_INCONS : ZIP_ER_NOZIP;
			}
			za->mode = 0; /* nothing to finalize */
			zip_close (za);
			return NULL;
		}
		a->n_existing = za->n_entries;
		if (za->mode == 1) {
			za->next_index = za->n_entries;
		}
	}
	if (errorp) {
		*errorp = 0;
	}
	return za;
fail_flags:
	if (errorp) {
		*errorp = -1;
	}
	free (a);
	return NULL;
}

/* otezip.c:1406-1440: temp-file trampoline */
zip_t *zip_open_from_source(zip_source_t *src, int flags, zip_error_t *error) {
	(void)error;
	if (!src) {
		return NULL;
	}
	char tmp[] = "/tmp/otezip_XXXXXX";
	mode_t old = umask (077);
	int fd = mkstemp (tmp);
	umask (old);
	if (fd < 0) {
		return NULL;
	}
	ssize_t w = write (fd, src->buf, (size_t)src->len);
	close (fd);
	if (w < 0 || (zip_uint64_t)w != src->len) {
		unlink (tmp);
		return NULL;
	}
	int err = 0;
	zip_t *za = zip_open (tmp, flags, &err);
	if (!za) {
		unlink (tmp);
	}
	return za;
}

static int finalize_archive(struct otz_archive *a);
static int zstd_frames(void);

int zip_close(zip_t *za) {
	struct otz_archive *a = priv (za);
	if (!is_valid (za) || !a) {
		free (za); /* otezip.c:1274-1277 */
		return -1;
	}
	int rc = 0;
	if (za->mode == 1) {
		rc = finalize_archive (a);
	}
	fclose (za->fp);
	for (zip_uint64_t i = 0; i < za->n_entries; i++) {
		free (za->entries[i].name);
	}
	if (a->pend) {
		for (zip_uint64_t i = 0; i < za->n_entries; i++) {
			if (a->pend[i].owned) {
				free (a->pend[i].buf);
			}
			wipe_free (a->pend[i].pw);
		}
		free (a->pend);
	}
	wipe_free (a->default_pw);
	free (a->aes);
	free (za->entries);
	free_windows (a);
	if (a->image) {
		otz_host_free (a->image);
	}
	free (a->last_status);
	free (a->lfh64);
	free (a->path);
	a->magic = 0;
	free (a);
	return rc;
}

zip_uint64_t zip_get_num_files(zip_t *za) {
	return za ? za->n_entries : 0u; /* otezip.c:1297-1299 */
}

zip_int64_t zip_name_locate(zip_t *za, const char *fname, zip_flags_t flags) {
	(void)flags;
	if (!is_valid (za) || !fname) {
		return -1;
	}
	for (zip_uint64_t i = 0; i < za->n_entries; i++) {
		if (!strcmp (za->entries[i].name, fname)) {
			return (zip_int64_t)i;
		}
	}
	return -1;
}

const char *zip_get_name(zip_t *za, zip_uint64_t index, zip_flags_t flags) {
	(void)flags;
	return (is_valid (za) && index < za->n_entries) ? za->entries[index].name : NULL;
}

void zip_stat_init(zip_stat_t *st) { /* otezip.c:1359-1371 */
	if (st) {
		memset (st, 0, sizeof (*st));
		st->index = ZIP_UINT64_MAX;
		st->mtime = (time_t)-1;
		st->comp_method = ZIP_CM_STORE;
	}
}

int zip_stat_index(zip_t *za, zip_uint64_t index, zip_flags_t flags, zip_stat_t *st) {
	(void)flags;
	if (!is_valid (za) || !st || index >= za->n_entries) {
		return -1;
	}
	const struct otezip_entry *e = &za->entries[index];
	zip_stat_init (st);
	st->name = e->name;
	st->index = index;
	st->size = e->uncomp_size;
	st->comp_size = e->comp_size;
	st->crc = e->crc32;
	st->comp_method = e->method;
	st->valid = ZIP_STAT_NAME | ZIP_STAT_INDEX | ZIP_STAT_SIZE | ZIP_STAT_COMP_SIZE | ZIP_STAT_CRC | ZIP_STAT_COMP_METHOD;
	return 0;
}

int zip_stat(zip_t *za, const char *fname, zip_flags_t flags, zip_stat_t *st) {
	zip_int64_t i = zip_name_locate (za, fname, flags);
	return i < 0 ? -1 : zip_stat_index (za, (zip_uint64_t)i, flags, st);
}

/* ---------------------------------------------------------------- read path: batched extract */

static uint64_t batch_budget(void) {
	const char *e = getenv ("OTEZIP_BATCH_BYTES");
	uint64_t v = e ? strtoull (e, NULL, 10) : 0;
	return v ? v : (4ULL << 30); /* decoded bytes per batch */
}

static void free_window(struct otz_window *w) {
	if (w->arena) {
		otz_host_free (w->arena);
	}
	free (w->ofs);
	free (w->status);
	free (w->crc);
	free (w);
}

static void free_windows(struct otz_archive *a) {
	struct otz_window *w = a->windows;
	while (w) {
		struct otz_window *n = w->next;
		if (w->refs) {
			/* zip_file_t handles still point into the arena.  In the reference every handle owns its buffer
			 * (otezip.c:1326-1331), so zf->data stays valid after zip_close: keep the window until its last handle closes */
			w->orphan = 1;
			w->next = NULL;
		} else {
			free_window (w);
		}
		w = n;
	}
	a->windows = NULL;
}

static void drop_idle_windows(struct otz_archive *a) {
	struct otz_window **pp = &a->windows;
	while (*pp) {
		struct otz_window *w = *pp;
		if (!w->current && w->refs == 0) {
			*pp = w->next;
			free_window (w);
		} else {
			pp = &w->next;
		}
	}
}

/* the zip-bomb rule of otezip.c:454-462, evaluated with the globals as they are NOW; an AES entry is judged by its
 * ciphertext, what the decoder reads */
static int bomb_rejects(const struct otz_archive *a, zip_uint64_t i) {
	const uint64_t comp = inner_comp (a, i);
	if (otezip_ignore_zipbomb || comp == 0) {
		return 0;
	}
	uint64_t allowed = comp * otezip_max_expansion_ratio + otezip_max_expansion_slack;
	return (uint64_t)a->pub.entries[i].uncomp_size > allowed;
}

static int load_image(struct otz_archive *a) {
	if (a->image) {
		return 0;
	}
	FILE *fp = a->pub.fp;
	if (fseek (fp, 0, SEEK_END) != 0) {
		return -1;
	}
	long fsz = ftell (fp);
	if (fsz < 0) {
		return -1;
	}
	void *p = NULL;
	if (otz_host_alloc ((uint64_t)fsz + 64, &p) != OTZ_SUCCESS) {
		fprintf (stderr, "otezip-b200: %s\n", otz_last_error ());
		return -1;
	}
	if (read_at (fp, 0, p, (size_t)fsz) != 0) {
		otz_host_free (p);
		return -1;
	}
	a->image = (uint8_t *)p;
	a->image_len = (uint64_t)fsz;
	return 0;
}

/* Chunk index of an entry (LFH extra field 'OZ'), validated against the directory values.  Returns the number of
 * chunks (>= 2) and points *csize at the u32 LE array inside the image, or 0 when the entry has no usable index. */
static uint32_t chunk_index_of(const struct otz_archive *a, const struct otezip_entry *e, uint32_t *chunk_bytes, const uint8_t **csize,
	uint64_t *data_ofs) {
	const uint64_t lfh_ofs = entry_lfh (&a->pub, (zip_uint64_t)(e - a->pub.entries));
	if (!index_enabled () || e->method != OTEZIP_METHOD_DEFLATE || lfh_ofs + 30 > a->image_len) {
		return 0;
	}
	const uint8_t *lfh = a->image + lfh_ofs;
	if (otezip_read_le32 (lfh) != SIG_LFH) {
		return 0;
	}
	const uint64_t nl = otezip_read_le16 (lfh + 26), xl = otezip_read_le16 (lfh + 28);
	const uint64_t xofs = lfh_ofs + 30 + nl;
	if (xofs + xl + e->comp_size > a->image_len) {
		return 0;
	}
	const uint8_t *x = a->image + xofs;
	for (uint64_t o = 0; o + 4 <= xl;) {
		const uint32_t id = otezip_read_le16 (x + o), sz = otezip_read_le16 (x + o + 2);
		if (o + 4 + sz > xl) {
			return 0;
		}
		if (id == OZ_EXTRA_ID && sz >= 12 && x[o + 4] == 1) {
			const uint32_t cb = otezip_read_le32 (x + o + 8), nc = otezip_read_le32 (x + o + 12);
			if (cb == 0 || cb > 65535 || nc < 2 || nc > OZ_EXTRA_MAX_CHUNKS || sz != 12 + 4 * nc ||
				(uint64_t)nc != ((uint64_t)e->uncomp_size + cb - 1) / cb) {
				return 0;
			}
			uint64_t sum = 0;
			for (uint32_t c = 0; c < nc; c++) {
				sum += otezip_read_le32 (x + o + 16 + 4 * c);
			}
			if (sum != e->comp_size) {
				return 0;
			}
			*chunk_bytes = cb;
			*csize = x + o + 16;
			*data_ofs = xofs + xl;
			return nc;
		}
		o += 4 + sz;
	}
	return 0;
}

/* Decode a batch starting at `index`: consecutive entries until the byte budget is reached.  Entries that carry
 * a chunk index become one parent row plus one row per chunk; if any chunk fails (or the CRC of the assembled
 * entry does not match) the entry is decoded again as one plain stream, so a wrong index can never change the
 * result the reference's sequential decoder would produce. */
/* What k_resolve would say about an entry, decided on the host from the image (the head of otezip_extract_entry,
 * otezip.c:403-487, in its order: LFH range and signature, payload range, zip-bomb rule, method, STORE size).  The
 * reference rejects such an entry BEFORE it allocates anything (otezip.c:454-462 precede the malloc at :470); here it
 * must not count towards the window's arena either: a crafted directory could otherwise claim gigabytes per entry. */
static int32_t host_precheck(const struct otz_archive *a, zip_uint64_t i, const char *pw) {
	const struct otezip_entry *e = &a->pub.entries[i];
	const uint64_t lfh = entry_lfh (&a->pub, i);
	const uint64_t len = a->image_len;
	if (lfh > len || len - lfh < 30) {
		return OTZ_ST_LFH_RANGE;
	}
	const uint8_t *h = a->image + lfh;
	if (otezip_read_le32 (h) != 0x04034b50u) {
		return OTZ_ST_LFH_SIG;
	}
	const uint64_t data = lfh + 30u + otezip_read_le16 (h + 26) + otezip_read_le16 (h + 28);
	if (data > len || (uint64_t)e->comp_size > MAX_PAYLOAD || (uint64_t)e->uncomp_size > MAX_PAYLOAD || data + e->comp_size > len) {
		return OTZ_ST_DATA_RANGE;
	}
	/* AES: the field must be usable and the payload hold salt, verification value and code; then the rules below apply
	 * to the inner stream (ciphertext size, actual method) as they would to the same bytes stored unencrypted */
	const struct otz_aesx *x = aes_of (a, i);
	if (x && !x->vendor) {
		return OTZ_ST_METHOD;
	}
	if (x && e->comp_size < AES_OVERHEAD (x->strength)) {
		return OTZ_ST_DATA_RANGE;
	}
	if (bomb_rejects (a, i)) {
		return OTZ_ST_ZIPBOMB;
	}
	const uint16_t method = x ? x->method : e->method;
	if (method == OTEZIP_METHOD_STORE) {
		if (inner_comp (a, i) != e->uncomp_size) {
			return OTZ_ST_STORE_SIZE;
		}
	} else if (method != OTEZIP_METHOD_DEFLATE && method != OTZ_M_DEFLATE64 && method != OTEZIP_METHOD_ZSTD && method != OTZ_M_XZ) {
		return OTZ_ST_METHOD;
	}
	if (x && !pw) {
		return OTZ_ST_NOPASSWD;
	}
	return OTZ_ST_OK;
}

/* Decode a batch starting at `index`: consecutive entries until the byte budget is reached.  Entries the host pre-check
 * rejects get their status here and a zero-length slice — they are not part of the device table, so neither the pinned
 * arena nor the device scratch is sized by what a directory merely claims.  Entries that carry a chunk index become one
 * parent row plus one row per chunk; a chunk row is only accepted in the shape this library writes (it ends byte
 * aligned behind an empty stored block, and only the last one holds the final block), and if any chunk fails or the CRC
 * of the assembled entry does not match, the entry is decoded again as one plain stream.  (The CRC comparison is the
 * backstop, not a proof: with otezip_ref_compat = 1 and otezip_verify_crc = 0 a crafted index whose chunks decode
 * cleanly AND collide on CRC-32 could still differ from the sequential decode; OTEZIP_NO_INDEX=1 ignores the index.) */
/* AES entries (method 99) are not rows of that table: they form a second batch on the first device (aes_batch).
 * pw_only != NULL: decode entry `index` alone with that password, into a window that is not cached (the caller owns it). */
static int aes_batch(struct otz_archive *a, struct otz_window *w, const uint32_t *ks, uint32_t m, const char *pw, otz_ctx *ctx);

static struct otz_window *run_window(struct otz_archive *a, zip_uint64_t index, const char *pw_only) {
	zip_t *za = &a->pub;
	otz_ctx **ctxs = NULL;
	const uint32_t n_ctx = otezip_b200_ctxs (&ctxs);
	if (!n_ctx || load_image (a) != 0) {
		return NULL;
	}
	const char *pw = pw_only ? pw_only : a->default_pw;
	const uint64_t budget = batch_budget ();
	/* A request BELOW every decoded window (reverse iteration, zip_name_locate-driven access) would otherwise decode a full
	 * window forward from each index it touches: start such a window up to half a budget earlier, so that the entries in
	 * front of the requested one are decoded with it. */
	int below_all = a->windows != NULL && !pw_only;
	zip_uint64_t lowest = za->n_entries;
	for (struct otz_window *p = a->windows; p; p = p->next) {
		below_all = below_all && index < p->first;
		lowest = p->first < lowest ? p->first : lowest;
	}
	if (below_all) {
		uint64_t back = ((uint64_t)za->entries[index].uncomp_size + 15) & ~15ULL;   /* (the requested entry itself must still fit) */
		while (index > 0) {
			const uint64_t sz = ((uint64_t)za->entries[index - 1].uncomp_size + 15) & ~15ULL;
			if (back + sz > budget / 2) {
				break;
			}
			back += sz;
			index--;
		}
	}
	zip_uint64_t last = index;
	uint64_t bytes = 0;
	while (last < za->n_entries) {
		if ((below_all && last >= lowest) || (pw_only && last > index)) {
			break;   /* (what follows is decoded already; or the entry is decoded on its own) */
		}
		const struct otezip_entry *e = &za->entries[last];
		uint64_t sz = host_precheck (a, last, pw) == OTZ_ST_OK ? ((uint64_t)e->uncomp_size + 15) & ~15ULL : 0;
		if (last > index && bytes + sz > budget) {
			break;
		}
		bytes += sz;
		last++;
	}
	const uint32_t n = (uint32_t)(last - index);
	/* rows of the device table: admitted entries first (compact), then their chunk rows */
	int32_t *pre = (int32_t *)calloc (n ? n : 1, sizeof (int32_t));
	uint32_t *rowof = (uint32_t *)calloc (n ? n : 1, sizeof (uint32_t));
	uint32_t *aes_ks = (uint32_t *)calloc (n ? n : 1, sizeof (uint32_t));
	if (!pre || !rowof || !aes_ks) {
		free (pre);
		free (rowof);
		free (aes_ks);
		return NULL;
	}
	uint32_t n_adm = 0, n_rows = 0, n_aes = 0;
	for (uint32_t k = 0; k < n; k++) {
		pre[k] = host_precheck (a, index + k, pw);
		rowof[k] = 0xFFFFFFFFu;
		if (pre[k] == OTZ_ST_OK && aes_of (a, index + k)) {
			aes_ks[n_aes++] = k;
		} else if (pre[k] == OTZ_ST_OK) {
			uint32_t cb;
			const uint8_t *cs;
			uint64_t dofs;
			rowof[k] = n_adm++;
			n_rows += chunk_index_of (a, &za->entries[index + k], &cb, &cs, &dofs);
		}
	}
	n_rows += n_adm;
	struct otz_window *w = (struct otz_window *)calloc (1, sizeof (*w));
	otz_entry *tab = (otz_entry *)calloc (n_rows ? n_rows : 1, sizeof (otz_entry));
	int32_t *row_status = (int32_t *)calloc (n_rows ? n_rows : 1, sizeof (int32_t));
	uint32_t *row_crc = (uint32_t *)calloc (n_rows ? n_rows : 1, sizeof (uint32_t));
	if (w) {
		w->ofs = (uint64_t *)calloc (n ? n : 1, sizeof (uint64_t));
		w->status = (int32_t *)calloc (n ? n : 1, sizeof (int32_t));
		w->crc = (uint32_t *)calloc (n ? n : 1, sizeof (uint32_t));
	}
	if (!w || !tab || !row_status || !row_crc || !w->ofs || !w->status || !w->crc) {
		if (w) {
			free_window (w);
		}
		free (tab);
		free (row_status);
		free (row_crc);
		free (pre);
		free (rowof);
		free (aes_ks);
		return NULL;
	}
	w->first = index;
	w->last = last;
	w->pw_gen = a->pw_gen;
	uint64_t out = 0;
	uint32_t next_row = n_adm; /* chunk rows follow the entry rows */
	for (uint32_t k = 0; k < n; k++) {
		const struct otezip_entry *e = &za->entries[index + k];
		w->ofs[k] = out;
		if (pre[k] != OTZ_ST_OK) {
			continue;
		}
		if (rowof[k] == 0xFFFFFFFFu) {   /* AES */
			out += ((uint64_t)e->uncomp_size + 15) & ~15ULL;
			continue;
		}
		otz_entry *t = &tab[rowof[k]];
		t->lfh_ofs = entry_lfh (za, index + k);
		t->out_ofs = out;
		t->comp_size = e->comp_size;
		t->uncomp_size = e->uncomp_size;
		t->crc32 = e->crc32;
		t->method = e->method;
		uint32_t cb = 0;
		const uint8_t *cs = NULL;
		uint64_t dofs = 0;
		const uint32_t nc = chunk_index_of (a, e, &cb, &cs, &dofs);
		if (nc) {
			t->flags = OTZ_EF_PARENT;
			uint64_t cofs = dofs, uofs = 0;
			for (uint32_t c = 0; c < nc; c++) {
				otz_entry *r = &tab[next_row++];
				const uint32_t csz = otezip_read_le32 (cs + 4 * c);
				r->lfh_ofs = cofs;
				r->out_ofs = out + uofs;
				r->comp_size = csz;
				r->uncomp_size = (uint32_t)((uint64_t)e->uncomp_size - uofs < cb ? (uint64_t)e->uncomp_size - uofs : cb);
				r->crc32 = rowof[k]; /* parent row */
				r->method = OTZ_M_DEFLATE;
				r->flags = (uint16_t)(OTZ_EF_CHUNK | (c + 1 == nc ? OTZ_EF_LAST_CHUNK : 0));
				cofs += csz;
				uofs += r->uncomp_size;
			}
		}
		out += ((uint64_t)e->uncomp_size + 15) & ~15ULL;
	}
	w->arena_len = out;
	void *arena = NULL;
	otz_extract_opts o;
	o.ignore_zipbomb = otezip_ignore_zipbomb;
	o.max_ratio = otezip_max_expansion_ratio;
	o.max_slack = otezip_max_expansion_slack;
	o.verify_only = 0;
	int rc = otz_host_alloc (out + 64, &arena);
	if (rc == OTZ_SUCCESS) {
		w->arena = (uint8_t *)arena;
		if (n_rows) {
			rc = otz_extract_host_multi (ctxs, n_ctx, a->image, a->image_len, tab, n_rows, &o, w->arena, out, row_crc, row_status, NULL);
		}
	}
	/* entries whose indexed decode did not come out clean are decoded again as plain streams */
	uint32_t n_redo = 0;
	for (uint32_t k = 0; rc == OTZ_SUCCESS && k < n_adm; k++) {
		if ((tab[k].flags & OTZ_EF_PARENT) && row_status[k] != OTZ_ST_OK) {
			n_redo++;
		}
	}
	if (rc == OTZ_SUCCESS && n_redo) {
		otz_entry *rt = (otz_entry *)calloc (n_redo, sizeof (otz_entry));
		int32_t *rs = (int32_t *)calloc (n_redo, sizeof (int32_t));
		uint32_t *rcv = (uint32_t *)calloc (n_redo, sizeof (uint32_t)), *map = (uint32_t *)calloc (n_redo, sizeof (uint32_t));
		if (rt && rs && rcv && map) {
			uint32_t m = 0;
			for (uint32_t k = 0; k < n_adm; k++) {
				if ((tab[k].flags & OTZ_EF_PARENT) && row_status[k] != OTZ_ST_OK) {
					rt[m] = tab[k];
					rt[m].flags = 0;
					map[m++] = k;
				}
			}
			rc = otz_extract_host_multi (ctxs, n_ctx, a->image, a->image_len, rt, n_redo, &o, w->arena, out, rcv, rs, NULL);
			for (uint32_t i = 0; rc == OTZ_SUCCESS && i < n_redo; i++) {
				row_status[map[i]] = rs[i];
				row_crc[map[i]] = rcv[i];
			}
		} else {
			rc = OTZ_ERR_NOMEM;
		}
		free (rt);
		free (rs);
		free (rcv);
		free (map);
	}
	for (uint32_t k = 0; k < n; k++) {
		const int plain = pre[k] == OTZ_ST_OK && rowof[k] != 0xFFFFFFFFu;
		w->status[k] = plain ? row_status[rowof[k]] : pre[k];
		w->crc[k] = plain ? row_crc[rowof[k]] : 0u;
	}
	if (rc == OTZ_SUCCESS && n_aes) {
		rc = aes_batch (a, w, aes_ks, n_aes, pw, ctxs[0]);
	}
	free (tab);
	free (row_status);
	free (row_crc);
	free (pre);
	free (rowof);
	free (aes_ks);
	if (rc != OTZ_SUCCESS) {
		fprintf (stderr, "otezip-b200: GPU extract failed: %s\n", otz_last_error ());
		free_window (w);
		return NULL;
	}
	if (pw_only) {
		w->orphan = 1;   /* not cached: freed by the last zip_fclose of its handles */
	} else {
		for (struct otz_window *p = a->windows; p; p = p->next) {
			p->current = 0;
		}
		w->current = 1;
		w->next = a->windows;
		a->windows = w;
		drop_idle_windows (a);
	}
	if (!a->last_status) {
		a->last_status = (int32_t *)malloc (za->n_entries * sizeof (int32_t));
		for (zip_uint64_t i = 0; a->last_status && i < za->n_entries; i++) {
			a->last_status[i] = -1;
		}
	}
	for (uint32_t k = 0; a->last_status && k < n; k++) {
		a->last_status[index + k] = w->status[k];
	}
	return w;
}

/* The AES entries ks[0..m) of window w (all past host_precheck): their payloads packed into one upload, each ciphertext
 * 16-byte aligned; otz_aes_open decrypts them into a plaintext image of synthetic local headers; that image is decoded
 * with the ordinary plan as an archive of plain entries (actual method, ciphertext size, directory CRC); the verdicts come
 * last.  NOPASSWD / WRONGPASSWD / AUTH override the decode's status, and only entries that pass the authentication code
 * are copied into the window's arena.  AE-2 stores no CRC (the code is the integrity check): its mismatch flag is dropped. */
static int aes_batch(struct otz_archive *a, struct otz_window *w, const uint32_t *ks, uint32_t m, const char *pw, otz_ctx *ctx) {
	zip_t *za = &a->pub;
	otz_aes_entry *rows = (otz_aes_entry *)calloc (m, sizeof (otz_aes_entry));
	otz_entry *tab = (otz_entry *)calloc (m, sizeof (otz_entry));
	int32_t *st = (int32_t *)calloc (m, sizeof (int32_t)), *verdict = (int32_t *)calloc (m, sizeof (int32_t));
	uint32_t *crc = (uint32_t *)calloc (m, sizeof (uint32_t));
	uint8_t *h_src = NULL;
	void *d_src = NULL, *d_plain = NULL, *d_out = NULL;
	otz_plan *plan = NULL;
	int rc = OTZ_ERR_NOMEM;
	uint64_t src_len = 0, plain_len = 0, out_len = 0;
	if (!rows || !tab || !st || !verdict || !crc) {
		goto out;
	}
	for (uint32_t j = 0; j < m; j++) {
		const zip_uint64_t i = w->first + ks[j];
		const struct otezip_entry *e = &za->entries[i];
		const struct otz_aesx *x = aes_of (a, i);
		const uint64_t pre = 4u + 4u * x->strength + 2u;          /* salt + verification value */
		rows[j].payload_ofs = ((src_len + pre + 15) & ~15ULL) - pre;
		rows[j].size = e->comp_size;
		rows[j].strength = x->strength;
		rows[j].password = 0;
		src_len = rows[j].payload_ofs + e->comp_size;
		rows[j].data_ofs = ((plain_len + 30 + 15) & ~15ULL) - 30;
		plain_len = rows[j].data_ofs + 30 + inner_comp (a, i);
		tab[j].lfh_ofs = rows[j].data_ofs;
		tab[j].out_ofs = out_len;
		tab[j].comp_size = (uint32_t)inner_comp (a, i);
		tab[j].uncomp_size = e->uncomp_size;
		tab[j].crc32 = e->crc32;
		tab[j].method = x->method;
		tab[j].flags = 0;
		out_len += ((uint64_t)e->uncomp_size + 15) & ~15ULL;
	}
	void *p = NULL;
	if ((rc = otz_host_alloc (src_len + 64, &p)) != OTZ_SUCCESS) {
		goto out;
	}
	h_src = (uint8_t *)p;
	for (uint32_t j = 0; j < m; j++) {
		const zip_uint64_t i = w->first + ks[j];
		const uint8_t *h = a->image + entry_lfh (za, i);
		const uint64_t data = entry_lfh (za, i) + 30u + otezip_read_le16 (h + 26) + otezip_read_le16 (h + 28);
		memcpy (h_src + rows[j].payload_ofs, a->image + data, rows[j].size);
	}
	otz_extract_opts o;
	o.ignore_zipbomb = otezip_ignore_zipbomb;
	o.max_ratio = otezip_max_expansion_ratio;
	o.max_slack = otezip_max_expansion_slack;
	o.verify_only = 0;
	if ((rc = otz_dev_alloc (ctx, src_len, &d_src)) != OTZ_SUCCESS || (rc = otz_dev_alloc (ctx, plain_len, &d_plain)) != OTZ_SUCCESS ||
		(rc = otz_dev_alloc (ctx, out_len, &d_out)) != OTZ_SUCCESS || (rc = otz_h2d (ctx, d_src, h_src, src_len)) != OTZ_SUCCESS ||
		(rc = otz_aes_open (ctx, (const uint8_t *)d_src, src_len, rows, m, &pw, 1, (uint8_t *)d_plain, plain_len)) != OTZ_SUCCESS) {
		goto out;
	}
	rc = otz_plan_create (ctx, tab, m, &o, &plan);
	if (rc == OTZ_SUCCESS) {
		rc = otz_extract_run (ctx, plan, (const uint8_t *)d_plain, plain_len, (uint8_t *)d_out, out_len);
	}
	if (rc == OTZ_SUCCESS) {
		rc = otz_extract_results (ctx, plan, crc, st);
	}
	{
		const int src = otz_aes_status (ctx, verdict);   /* (always collected: it joins the side stream and clears the keys) */
		rc = rc == OTZ_SUCCESS ? src : rc;
	}
	for (uint32_t j = 0; rc == OTZ_SUCCESS && j < m; j++) {
		const zip_uint64_t i = w->first + ks[j];
		int32_t s = st[j];
		if (verdict[j] != OTZ_ST_OK) {
			s = verdict[j];
		} else if (aes_of (a, i)->vendor == 2) {
			s &= ~OTZ_STF_CRC_MISMATCH;
		}
		w->status[ks[j]] = s;
		w->crc[ks[j]] = verdict[j] == OTZ_ST_OK ? crc[j] : 0u;
	}
	/* one copy per run of authenticated entries that lie at the same distances in the device output and in the arena
	 * (consecutive AES entries of the window, or separated only by rejected ones, whose slices are empty) */
	for (uint32_t j = 0; rc == OTZ_SUCCESS && j < m;) {
		if (verdict[j] != OTZ_ST_OK) {
			j++;
			continue;
		}
		uint32_t e = j + 1;
		while (e < m && verdict[e] == OTZ_ST_OK && w->ofs[ks[e]] - w->ofs[ks[j]] == tab[e].out_ofs - tab[j].out_ofs) {
			e++;
		}
		const uint64_t bytes = tab[e - 1].out_ofs + tab[e - 1].uncomp_size - tab[j].out_ofs;
		if (bytes) {
			rc = otz_d2h (ctx, w->arena + w->ofs[ks[j]], (const uint8_t *)d_out + tab[j].out_ofs, bytes);
		}
		j = e;
	}
	if (rc == OTZ_SUCCESS) {
		rc = otz_sync (ctx);
	}
out:
	if (plan) {
		otz_plan_destroy (ctx, plan);
	}
	if (d_src) {
		otz_dev_free (ctx, d_src);
	}
	if (d_plain) {
		otz_dev_memset (ctx, d_plain, 0, plain_len);   /* (the plaintext does not outlive the batch on the device) */
		otz_sync (ctx);
		otz_dev_free (ctx, d_plain);
	}
	if (d_out) {
		otz_dev_memset (ctx, d_out, 0, out_len);   /* (nor its decode, which includes entries that failed authentication) */
		otz_sync (ctx);
		otz_dev_free (ctx, d_out);
	}
	if (h_src) {
		otz_host_free (h_src);
	}
	free (rows);
	free (tab);
	free (st);
	free (verdict);
	free (crc);
	return rc;
}

int otezip_b200_entry_status(zip_t *za, zip_uint64_t index) {
	struct otz_archive *a = priv (za);
	if (!a || !a->last_status || index >= za->n_entries) {
		return -1;
	}
	return a->last_status[index];
}

/* The handle of entry `index` from window w, or NULL when the current globals reject its status. */
static zip_file_t *hand_out(struct otz_archive *a, struct otz_window *w, zip_uint64_t index) {
	struct otezip_entry *e = &a->pub.entries[index];
	const struct otz_aesx *x = aes_of (a, index);
	const uint32_t k = (uint32_t)(index - w->first);
	int32_t st = w->status[k];
	if (OTZ_ST_CODE (st) == OTZ_ST_OK && bomb_rejects (a, index)) {
		st = OTZ_ST_ZIPBOMB; /* the guard tightened since the batch ran */
	}
	if (OTZ_ST_CODE (st) == OTZ_ST_ZIPBOMB) { /* otezip.c:459, verbatim */
		fprintf (stderr, "mzip: entry '%s' claims huge uncompressed size (%u), rejecting to avoid zipbomb\n",
			e->name ? e->name : "<unknown>", e->uncomp_size);
		return NULL;
	}
	const uint16_t method = x ? x->method : e->method;
	if (OTZ_ST_CODE (st) != OTZ_ST_OK || (otezip_ref_compat && (st & OTZ_STF_REF_EOB) && !(method == OTEZIP_METHOD_ZSTD && zstd_frames ()))) {
		return NULL;
	}
	if (st & OTZ_STF_CRC_MISMATCH) { /* otezip.c:669-678 */
		if (otezip_verify_crc) {
			return NULL;
		}
		fprintf (stderr, "Warning: CRC mismatch for '%s' (expected 0x%08x, got 0x%08x)\n", e->name ? e->name : "<unknown>", e->crc32,
			w->crc[k]);
	}
	struct otz_file *f = (struct otz_file *)calloc (1, sizeof (*f));
	if (!f) {
		return NULL;
	}
	f->pub.data = w->arena + w->ofs[k];
	f->pub.size = e->uncomp_size;
	f->pub.pos = 0;
	f->win = w;
	w->refs++;
	return &f->pub;
}

/* otezip.c:1315-1334 + :399-684 */
zip_file_t *zip_fopen_index(zip_t *za, zip_uint64_t index, zip_flags_t flags) {
	(void)flags;
	struct otz_archive *a = priv (za);
	if (!is_valid (za) || !a || index >= za->n_entries) {
		return NULL;
	}
	if (za->mode == 1 && (index >= a->n_existing || (a->pend && a->pend[index].dirty))) {
		return NULL; /* queued, not yet written */
	}
	struct otz_window *w = NULL;
	for (struct otz_window *p = a->windows; p; p = p->next) {
		if (index >= p->first && index < p->last) {
			w = p;
			break;
		}
	}
	/* a batch decoded under other zip-bomb globals may have skipped this entry, and an AES entry decoded under another
	 * default password must not be handed out: decide again */
	if (w) {
		int st = w->status[index - w->first];
		if ((OTZ_ST_CODE (st) == OTZ_ST_ZIPBOMB && !bomb_rejects (a, index)) || (aes_of (a, index) && w->pw_gen != a->pw_gen)) {
			w = NULL;
		}
	}
	if (!w) {
		w = run_window (a, index, NULL);
		if (!w) {
			return NULL;
		}
	}
	return hand_out (a, w, index);
}

/* libzip: open an entry with this password instead of the default one.  The result is bound to the password: unless it is
 * the default password (whose results are cached), the entry is decoded again, on its own. */
zip_file_t *zip_fopen_index_encrypted(zip_t *za, zip_uint64_t index, zip_flags_t flags, const char *password) {
	struct otz_archive *a = priv (za);
	if (!is_valid (za) || !a || index >= za->n_entries) {
		return NULL;
	}
	if (!password || !aes_of (a, index) || (a->default_pw && !strcmp (password, a->default_pw))) {
		return zip_fopen_index (za, index, flags);
	}
	if (za->mode == 1 && (index >= a->n_existing || (a->pend && a->pend[index].dirty))) {
		return NULL;
	}
	struct otz_window *w = run_window (a, index, password);
	if (!w) {
		return NULL;
	}
	zip_file_t *f = hand_out (a, w, index);
	if (!f) {
		free_window (w);
	}
	return f;
}

int zip_set_default_password(zip_t *za, const char *password) {
	struct otz_archive *a = priv (za);
	if (!is_valid (za) || !a) {
		return -1;
	}
	char *copy = password ? strdup (password) : NULL;
	if (password && !copy) {
		return -1;
	}
	wipe_free (a->default_pw);
	a->default_pw = copy;
	a->pw_gen++;   /* cached AES results belong to the old password */
	return 0;
}

int zip_compression_method_supported(zip_int32_t method, int compress) {
	if (method == ZIP_CM_STORE || method == ZIP_CM_DEFLATE || method == OTEZIP_METHOD_ZSTD) {
		return 1;
	}
	return !compress && (method == ZIP_CM_DEFLATE64 || method == ZIP_CM_XZ);   /* Deflate64 and XZ are read, never written */
}

int zip_encryption_method_supported(zip_uint16_t method, int encode) {
	(void)encode;
	return method == ZIP_EM_NONE || method == ZIP_EM_AES_128 || method == ZIP_EM_AES_192 || method == ZIP_EM_AES_256;
}

/* libzip: encrypt an entry added or replaced in this session (as zip_set_file_compression, entries already on disk are
 * refused); ZIP_EM_NONE undoes it.  password NULL: the default password at zip_close. */
int zip_file_set_encryption(zip_t *za, zip_uint64_t index, zip_uint16_t method, const char *password) {
	struct otz_archive *a = priv (za);
	if (!is_valid (za) || !a || index >= za->n_entries || za->mode != 1 || !a->pend || !zip_encryption_method_supported (method, 1)) {
		return -1;
	}
	if (index < a->n_existing && !a->pend[index].dirty) {
		return -1;
	}
	char *copy = password ? strdup (password) : NULL;
	if (password && !copy) {
		return -1;
	}
	wipe_free (a->pend[index].pw);
	a->pend[index].pw = method == ZIP_EM_NONE ? NULL : copy;
	if (method == ZIP_EM_NONE) {
		wipe_free (copy);
	}
	a->pend[index].enc = method == ZIP_EM_NONE ? 0 : (uint16_t)(method & 0xFF);
	return 0;
}

int zip_fclose(zip_file_t *zf) { /* otezip.c:1336-1343: the library owns zf->data */
	if (!zf) {
		return -1;
	}
	struct otz_file *f = (struct otz_file *)zf;
	if (f->win && f->win->refs) {
		f->win->refs--;
		if (!f->win->refs && f->win->orphan) {
			free_window (f->win);
		}
	}
	free (f->own);
	free (f);
	return 0;
}

zip_int64_t zip_fread(zip_file_t *zf, void *buf, zip_uint64_t nbytes) { /* otezip.c:1345-1357 */
	if (!zf || !buf) {
		return -1;
	}
	if (zf->pos >= zf->size) {
		return 0;
	}
	zip_uint64_t left = zf->size - zf->pos;
	zip_uint64_t n = nbytes < left ? nbytes : left;
	memcpy (buf, zf->data + zf->pos, n);
	zf->pos += n;
	return (zip_int64_t)n;
}

/* ---------------------------------------------------------------- write path: queue, then one GPU batch */

zip_source_t *zip_source_buffer(zip_t *za, const void *data, zip_uint64_t len, int freep) { /* otezip.c:1592-1599 */
	(void)za;
	zip_source_t *s = (zip_source_t *)malloc (sizeof (*s));
	if (s) {
		s->buf = data;
		s->len = len;
		s->freep = freep;
	}
	return s;
}

zip_source_t *zip_source_buffer_create(const void *data, zip_uint64_t len, int freep, zip_error_t *error) {
	(void)error;
	return zip_source_buffer (NULL, data, len, freep);
}

void zip_source_free(zip_source_t *src) { /* otezip.c:1606-1614 */
	if (src) {
		if (src->freep && src->buf) {
			free ((void *)src->buf);
		}
		free (src);
	}
}

/* Take the bytes of a source for later compression.  freep: the library owns the caller's buffer from
 * now on (otezip.c:1172-1174 frees it right away; here it lives until zip_close).  !freep: the
 * reference has consumed the bytes when zip_file_add returns, so the caller may reuse the buffer:
 * keep a private copy. */
static int take_source(struct otz_pending *p, zip_source_t *src) {
	p->len = src->len;
	if (src->freep || src->len == 0) {
		p->buf = (void *)src->buf;
		p->owned = src->freep;
		return 0;
	}
	p->buf = malloc ((size_t)src->len);
	if (!p->buf) {
		return -1;
	}
	memcpy (p->buf, src->buf, (size_t)src->len);
	p->owned = 1;
	return 0;
}

/* otezip.c:1079-1183, with compression deferred to zip_close */
zip_int64_t zip_file_add(zip_t *za, const char *name, zip_source_t *src, zip_flags_t flags) {
	(void)flags;
	struct otz_archive *a = priv (za);
	if (!a || !name || !src || za->mode != 1) {
		return -1;
	}
	size_t nlen = strlen (name);
	if (nlen > MAX_FIELD_LEN || (uint64_t)src->len > MAX_PAYLOAD) {
		return -1;
	}
	struct otezip_entry *ne = (struct otezip_entry *)realloc (za->entries, (za->n_entries + 1) * sizeof (*ne));
	if (!ne) {
		return -1;
	}
	za->entries = ne;
	struct otz_pending *np = (struct otz_pending *)realloc (a->pend, (za->n_entries + 1) * sizeof (*np));
	if (!np) {
		return -1;
	}
	if (!a->pend) {
		memset (np, 0, za->n_entries * sizeof (*np));
	}
	a->pend = np;
	struct otezip_entry *e = &za->entries[za->n_entries];
	struct otz_pending *p = &a->pend[za->n_entries];
	memset (e, 0, sizeof (*e));
	memset (p, 0, sizeof (*p));
	e->name = (char *)malloc (nlen + 1);
	if (!e->name) {
		return -1;
	}
	memcpy (e->name, name, nlen + 1);
	e->method = za->default_method > 0 ? za->default_method : 0; /* otezip.c:1109-1114 */
	e->uncomp_size = (uint32_t)src->len;
	dos_now (&e->file_time, &e->file_date);                      /* otezip.c:1127 */
	e->external_attr = 0100644u << 16;                            /* otezip.c:1130 */
	if (take_source (p, src) != 0) {
		free (e->name);
		return -1;
	}
	p->dirty = 1;
	free (src); /* consumed, otezip.c:1175 */
	zip_uint64_t idx = za->n_entries++;
	za->next_index = za->n_entries;
	return (zip_int64_t)idx;
}

zip_int64_t zip_add(zip_t *za, const char *name, zip_source_t *src) {
	return zip_file_add (za, name, src, 0);
}

/* otezip.c:1186-1237 — the method now really applies, because nothing has been compressed yet */
int zip_set_file_compression(zip_t *za, zip_uint64_t index, zip_int32_t comp, zip_uint32_t comp_flags) {
	struct otz_archive *a = priv (za);
	if (!is_valid (za) || !a || index >= za->n_entries || za->mode != 1) {
		return -1;
	}
	if (comp != OTEZIP_METHOD_STORE && comp != OTEZIP_METHOD_DEFLATE && comp != OTEZIP_METHOD_ZSTD) {
		return -1;
	}
	if (index < a->n_existing && !(a->pend && a->pend[index].dirty)) {
		return -1; /* already on disk: relabelling would corrupt it (the reference's F4 bug) */
	}
	za->entries[index].method = (uint16_t)comp;
	/* comp_flags is libzip's compression level (0 = default, 1 = fastest .. 9 = best; the reference ignores it,
	 * otezip.c:1186): 1-3 select the compressor's single-candidate parse (OTZ_M_FAST), 7-9 the best level of DEFLATE
	 * (OTZ_M_BEST: hash chains searched at every position; method 93 takes them as the default), 0 and 4-6 the
	 * default eight-way search */
	if (a->pend) {
		a->pend[index].level = comp_flags;
	}
	return 0;
}

/* otezip.c:1617-1663: new bytes for an entry — one added in this session or one that is already in the archive
 * (append mode).  The reference compresses and writes them at once and leaves `src` to the caller; here they are
 * queued like every other source (always as a private copy, since the caller keeps `src`) and written by zip_close
 * behind the existing data; the central directory then points at the new copy, as in the reference. */
int zip_file_replace(zip_t *za, zip_uint64_t index, zip_source_t *src, zip_flags_t flags) {
	(void)flags;
	struct otz_archive *a = priv (za);
	if (!is_valid (za) || !a || !src || za->mode != 1 || index >= za->n_entries || (uint64_t)src->len > MAX_PAYLOAD) {
		return -1;
	}
	if (!a->pend) {
		a->pend = (struct otz_pending *)calloc (za->n_entries, sizeof (*a->pend));
		if (!a->pend) {
			return -1;
		}
	}
	struct otz_pending np;
	memset (&np, 0, sizeof (np));
	np.len = src->len;
	if (src->len) {
		np.buf = malloc ((size_t)src->len);
		if (!np.buf) {
			return -1;
		}
		memcpy (np.buf, src->buf, (size_t)src->len);
		np.owned = 1;
	}
	np.dirty = 1;
	np.level = a->pend[index].level; /* the level asked for with zip_set_file_compression stays with the entry */
	np.enc = a->pend[index].enc;   /* and so does the encryption asked for with zip_file_set_encryption */
	np.pw = a->pend[index].pw;
	if (a->pend[index].owned) {
		free (a->pend[index].buf);
	}
	a->pend[index] = np;
	za->entries[index].uncomp_size = (uint32_t)src->len;
	if (za->entries[index].method != OTEZIP_METHOD_STORE && za->entries[index].method != OTEZIP_METHOD_DEFLATE &&
		za->entries[index].method != OTEZIP_METHOD_ZSTD) {
		za->entries[index].method = OTEZIP_METHOD_STORE; /* otezip_compress_data's default arm (otezip.c:803-812) */
	}
	return 0;
}

int zip_replace(zip_t *za, zip_uint64_t index, zip_source_t *src) {
	return zip_file_replace (za, index, src, 0);
}

/* otezip.c:1443-1491 */
/* 1: method 93 means real Zstandard frames on both paths (SURVEY.md §8f rank 3) — zip_close compresses entries whose
 * method is ZSTD with the GPU Zstandard encoder (k_zstd_enc.cuh) instead of ending up at STORE as the reference's raw-block
 * stub always does (otezip.c:894-899), and zip_fopen_index hands out the bytes of real frames although the reference's
 * reader rejects them (F3).  Default 0: the reference's observable behaviour. */
static int zstd_frames(void) {
	const char *e = getenv ("OTEZIP_ZSTD_FRAMES");
	return otezip_zstd_frames || (e && *e && *e != '0');
}

static int streaming_layout(void) {
	const char *e = getenv ("OTEZIP_DATA_DESCRIPTORS");
	return otezip_write_data_descriptors || (e && *e && *e != '0');
}

static int write_lfh(FILE *fp, const struct otezip_entry *e, const uint8_t *extra, uint16_t extra_len, int streaming, int encrypted) {
	uint8_t h[30];
	uint16_t t, d;
	size_t nl = strlen (e->name);
	dos_now (&t, &d); /* the reference re-samples the clock here, otezip.c:1464-1467 */
	otezip_write_le32 (h, SIG_LFH);
	otezip_write_le16 (h + 4, 20);
	otezip_write_le16 (h + 6, (streaming ? 0x0008 : 0) | (encrypted ? 0x0001 : 0)); /* bit 3: CRC and sizes follow the payload (APPNOTE 4.3.9) */
	otezip_write_le16 (h + 8, e->method);
	otezip_write_le16 (h + 10, t);
	otezip_write_le16 (h + 12, d);
	otezip_write_le32 (h + 14, streaming ? 0 : e->crc32);
	otezip_write_le32 (h + 18, streaming ? 0 : e->comp_size);
	otezip_write_le32 (h + 22, streaming ? 0 : e->uncomp_size);
	otezip_write_le16 (h + 26, (uint16_t)nl);
	otezip_write_le16 (h + 28, extra_len);
	return fwrite (h, 1, 30, fp) == 30 && fwrite (e->name, 1, nl, fp) == nl &&
			(!extra_len || fwrite (extra, 1, extra_len, fp) == extra_len)
		? 0
		: -1;
}

/* otezip.c:1494-1558; a local header beyond 4 GiB is written as the ZIP64 escape + extended information field */
/* data descriptor behind the payload of a streamed entry (APPNOTE 4.3.9, with the customary signature) */
static int write_descriptor(FILE *fp, const struct otezip_entry *e) {
	uint8_t h[16];
	otezip_write_le32 (h, 0x08074b50u);
	otezip_write_le32 (h + 4, e->crc32);
	otezip_write_le32 (h + 8, e->comp_size);
	otezip_write_le32 (h + 12, e->uncomp_size);
	return fwrite (h, 1, 16, fp) == 16 ? 0 : -1;
}

/* the 0x9901 field of an AES entry (11 bytes) */
static void aes_extra(uint8_t *x, const struct otz_aesx *ax) {
	otezip_write_le16 (x, AES_EXTRA_ID);
	otezip_write_le16 (x + 2, 7);
	otezip_write_le16 (x + 4, ax->vendor);
	x[6] = 'A';
	x[7] = 'E';
	x[8] = ax->strength;
	otezip_write_le16 (x + 9, ax->method);
}

static uint32_t write_cdh(FILE *fp, const struct otezip_entry *e, uint64_t lfh_ofs, int streaming, const struct otz_aesx *ax) {
	uint8_t h[46], x[12 + 11];
	size_t nl = strlen (e->name);
	const int z64 = lfh_ofs >= 0xFFFFFFFFULL;
	const int enc = ax && ax->vendor;
	const uint16_t xl = (uint16_t)((z64 ? 12 : 0) + (enc ? 11 : 0));
	memset (h, 0, sizeof (h));
	otezip_write_le32 (h, SIG_CDH);
	otezip_write_le16 (h + 4, 0x031e);
	otezip_write_le16 (h + 6, z64 ? 45 : 20);
	otezip_write_le16 (h + 8, (streaming ? 0x0008 : 0) | (enc ? 0x0001 : 0));
	otezip_write_le16 (h + 10, e->method);
	otezip_write_le16 (h + 12, e->file_time);
	otezip_write_le16 (h + 14, e->file_date);
	otezip_write_le32 (h + 16, e->crc32);
	otezip_write_le32 (h + 20, e->comp_size);
	otezip_write_le32 (h + 24, e->uncomp_size);
	otezip_write_le16 (h + 28, (uint16_t)nl);
	otezip_write_le16 (h + 30, xl);
	otezip_write_le32 (h + 38, e->external_attr);
	otezip_write_le32 (h + 42, z64 ? 0xFFFFFFFFu : (uint32_t)lfh_ofs);
	fwrite (h, 1, 46, fp);
	fwrite (e->name, 1, nl, fp);
	if (z64) {
		otezip_write_le16 (x, 0x0001);
		otezip_write_le16 (x + 2, 8);
		otezip_write_le32 (x + 4, (uint32_t)lfh_ofs);
		otezip_write_le32 (x + 8, (uint32_t)(lfh_ofs >> 32));
	}
	if (enc) {
		aes_extra (x + (z64 ? 12 : 0), ax);
	}
	if (xl) {
		fwrite (x, 1, xl, fp);
	}
	return (uint32_t)(46 + nl + xl);
}

/* The encrypted entries of a write batch: sealed on the device straight from the compressor's dense arena (otz_aes_seal), then
 * fetched.  *sealed[sofs[k] ..] holds salt | verification value | ciphertext | code of new entry k (sofs[k] = ~0 for entries
 * that are not encrypted).  Salts come from getrandom(2), one per entry; without random bytes nothing is written. */
#define SEAL_BATCH 65534u
static int seal_entries(struct otz_archive *a, otz_ctx *ctx, otz_deflate_job *job, const zip_uint64_t *idx, zip_uint64_t n_new,
	const uint64_t *out_ofs, const uint32_t *out_size, uint64_t out_total, uint8_t **sealed, uint64_t *sofs) {
	zip_uint64_t m = 0;
	uint64_t len = 0;
	for (zip_uint64_t k = 0; k < n_new; k++) {
		sofs[k] = ~0ULL;
		const struct otz_pending *p = &a->pend[idx[k]];
		if (p->enc) {
			const uint64_t pre = 4u + 4u * p->enc + 2u;
			sofs[k] = ((len + pre + 15) & ~15ULL) - pre;
			len = sofs[k] + out_size[k] + AES_OVERHEAD (p->enc);
			m++;
		}
	}
	otz_aes_entry *rows = (otz_aes_entry *)calloc (m, sizeof (*rows));
	const char **pws = (const char **)calloc (m, sizeof (*pws));
	const char **uniq = (const char **)calloc (m < SEAL_BATCH ? m + 1 : SEAL_BATCH, sizeof (*uniq));
	uint8_t *salts = (uint8_t *)calloc (m, 16);
	void *d_out = NULL, *h = NULL;
	int rc = -1;
	if (!rows || !pws || !uniq || !salts) {
		goto out;
	}
	uint32_t j = 0;
	for (zip_uint64_t k = 0; k < n_new; k++) {
		const struct otz_pending *p = &a->pend[idx[k]];
		if (!p->enc) {
			continue;
		}
		pws[j] = p->pw ? p->pw : a->default_pw;
		if (!pws[j]) {
			fprintf (stderr, "otezip-b200: no password for the encrypted entry '%s'\n", a->pub.entries[idx[k]].name);
			goto out;
		}
		rows[j].payload_ofs = sofs[k];
		rows[j].data_ofs = out_ofs[k];
		rows[j].size = out_size[k];
		rows[j].strength = p->enc;
		j++;
	}
	for (uint64_t got = 0; got < 16 * m;) {
		const ssize_t r = getrandom (salts + got, 16 * m - got, 0);
		if (r <= 0 && errno != EINTR) {
			fprintf (stderr, "otezip-b200: no random bytes for the salts: %s\n", strerror (errno));
			goto out;
		}
		got += r > 0 ? (uint64_t)r : 0;
	}
	if (otz_host_alloc (len + 64, &h) != OTZ_SUCCESS || otz_dev_alloc (ctx, len, &d_out) != OTZ_SUCCESS) {
		fprintf (stderr, "otezip-b200: %s\n", otz_last_error ());
		goto out;
	}
	/* One otz_aes_seal per SEAL_BATCH entries (a call indexes at most 65,534 passwords).  Its password list holds each
	 * distinct password once: an entry reuses the slot of the previous entry's password, or of any earlier one while the
	 * list is short; otherwise (many per-entry passwords) it gets a slot of its own. */
	for (zip_uint64_t b = 0; b < m; b += SEAL_BATCH) {
		const uint32_t nb = (uint32_t)(m - b < SEAL_BATCH ? m - b : SEAL_BATCH);
		uint32_t n_pw = 0;
		for (uint32_t q = 0; q < nb; q++) {
			const char *pw = pws[b + q];
			uint32_t slot = n_pw;
			if (n_pw && (uniq[n_pw - 1] == pw || !strcmp (uniq[n_pw - 1], pw))) {
				slot = n_pw - 1;
			} else if (n_pw <= 64) {
				for (uint32_t u = 0; u < n_pw; u++) {
					if (!strcmp (uniq[u], pw)) {
						slot = u;
						break;
					}
				}
			}
			if (slot == n_pw) {
				uniq[n_pw++] = pw;
			}
			rows[b + q].password = (uint16_t)slot;
		}
		if (otz_aes_seal (ctx, otz_deflate_device_output (job), out_total, rows + b, nb, salts + 16 * b, uniq, n_pw, (uint8_t *)d_out, len) !=
			OTZ_SUCCESS) {
			fprintf (stderr, "otezip-b200: GPU encrypt failed: %s\n", otz_last_error ());
			goto out;
		}
	}
	if (otz_d2h (ctx, h, d_out, len) != OTZ_SUCCESS || otz_sync (ctx) != OTZ_SUCCESS) {
		fprintf (stderr, "otezip-b200: GPU encrypt failed: %s\n", otz_last_error ());
		goto out;
	}
	*sealed = (uint8_t *)h;
	h = NULL;
	rc = 0;
out:
	if (d_out) {
		otz_dev_free (ctx, d_out);
	}
	if (h) {
		otz_host_free (h);
	}
	if (salts) {
		memset (salts, 0, 16 * m);
	}
	free (salts);
	free (pws);
	free (uniq);
	free (rows);
	return rc;
}

/* zip_close of a written archive: one GPU batch (CRC + DEFLATE/STORE decision), then LFH+payload per
 * entry in add order, the central directory and the EOCD (otezip.c:1240-1271, :1561-1590). */
static int finalize_archive(struct otz_archive *a) {
	zip_t *za = &a->pub;
	const int streaming = streaming_layout ();
	/* the entries to write: replaced existing ones and everything added in this session, in index order */
	zip_uint64_t n_new = 0;
	zip_uint64_t *idx = (zip_uint64_t *)calloc (za->n_entries ? za->n_entries : 1, sizeof (zip_uint64_t));
	if (!idx) {
		return -1;
	}
	for (zip_uint64_t i = 0; i < za->n_entries; i++) {
		if (i >= a->n_existing || (a->pend && a->pend[i].dirty)) {
			idx[n_new++] = i;
		}
	}
	uint64_t *in_ofs = NULL, *out_ofs = NULL, *sofs = NULL;
	uint8_t *sealed = NULL;
	uint32_t *in_len = NULL, *out_size = NULL, *crc = NULL;
	uint16_t *method = NULL, *method_out = NULL;
	uint8_t *in = NULL, *out = NULL;
	int rc = -1;
	uint64_t pos = a->n_existing ? a->append_ofs : 0;
	if (fseek (za->fp, (long)pos, SEEK_SET) != 0) {
		free (idx);
		return -1;
	}
	if (za->n_entries > a->aes_cap) {
		struct otz_aesx *na = (struct otz_aesx *)realloc (a->aes, za->n_entries * sizeof (*na));
		if (!na) {
			free (idx);
			return -1;
		}
		memset (na + a->aes_cap, 0, (za->n_entries - a->aes_cap) * sizeof (*na));
		a->aes = na;
		a->aes_cap = za->n_entries;
	}
	if (za->n_entries > a->lfh64_cap) {
		uint64_t *nl64 = (uint64_t *)realloc (a->lfh64, za->n_entries * sizeof (uint64_t));
		if (!nl64) {
			free (idx);
			return -1;
		}
		a->lfh64 = nl64;
		a->lfh64_cap = za->n_entries;
	}
	if (n_new) {
		otz_ctx *ctx = otezip_b200_ctx ();
		if (!ctx) {
			free (idx);
			return -1;
		}
		in_ofs = (uint64_t *)calloc (n_new, 8);
		out_ofs = (uint64_t *)calloc (n_new, 8);
		in_len = (uint32_t *)calloc (n_new, 4);
		out_size = (uint32_t *)calloc (n_new, 4);
		crc = (uint32_t *)calloc (n_new, 4);
		method = (uint16_t *)calloc (n_new, 2);
		method_out = (uint16_t *)calloc (n_new, 2);
		sofs = (uint64_t *)calloc (n_new, 8);
		if (!in_ofs || !out_ofs || !in_len || !out_size || !crc || !method || !method_out || !sofs) {
			goto done;
		}
		uint64_t total = 0;
		for (zip_uint64_t k = 0; k < n_new; k++) {
			const struct otezip_entry *e = &za->entries[idx[k]];
			in_ofs[k] = total;
			in_len[k] = (uint32_t)a->pend[idx[k]].len;
			/* method 93: the reference's writer cannot produce a stream its reader accepts and always falls
			 * back to STORE (zstd.inc.c:269, otezip.c:894-899; SURVEY.md F3) — same result here */
			method[k] = e->method == OTEZIP_METHOD_DEFLATE ? OTZ_M_DEFLATE : (e->method == OTEZIP_METHOD_ZSTD && zstd_frames ()) ? OTZ_M_ZSTD : OTZ_M_STORE;
			const uint32_t level = a->pend[idx[k]].level;
			if (level >= 1 && level <= 3 && method[k] != OTZ_M_STORE) {
				method[k] |= OTZ_M_FAST;
			} else if (level >= 7 && level <= 9 && method[k] == OTZ_M_DEFLATE) {
				method[k] |= OTZ_M_BEST;
			}
			total += ((uint64_t)in_len[k] + 15) & ~15ULL;
		}
		void *pin = NULL, *pout = NULL;
		if (otz_host_alloc (total + 64, &pin) != OTZ_SUCCESS || otz_host_alloc (total + 64, &pout) != OTZ_SUCCESS) {
			fprintf (stderr, "otezip-b200: %s\n", otz_last_error ());
			if (pin) {
				otz_host_free (pin);
			}
			goto done;
		}
		in = (uint8_t *)pin;
		out = (uint8_t *)pout;
		for (zip_uint64_t k = 0; k < n_new; k++) {
			if (in_len[k]) {
				memcpy (in + in_ofs[k], a->pend[idx[k]].buf, in_len[k]);
			}
		}
		uint64_t out_total = 0;
		otz_deflate_job *job = NULL;
		void *d_in = NULL;
		uint32_t *first_chunk = (uint32_t *)calloc (n_new, 4), *n_chunks = (uint32_t *)calloc (n_new, 4), *csize = NULL;
		uint32_t chunk_bytes = 0;
		int ok = first_chunk && n_chunks && otz_deflate_plan (ctx, in_ofs, in_len, method, (uint32_t)n_new, &job) == OTZ_SUCCESS &&
			otz_dev_alloc (ctx, total, &d_in) == OTZ_SUCCESS && otz_h2d (ctx, d_in, in, total) == OTZ_SUCCESS &&
			otz_deflate_run (ctx, job, (const uint8_t *)d_in, total) == OTZ_SUCCESS &&
			otz_deflate_results (ctx, job, out_ofs, out_size, crc, method_out, &out_total) == OTZ_SUCCESS && out_total <= total &&
			otz_deflate_fetch (ctx, job, out, out_total) == OTZ_SUCCESS;
		if (ok) {
			int nc_total = otz_deflate_chunks (ctx, job, first_chunk, n_chunks, NULL, 0, &chunk_bytes);
			csize = nc_total > 0 ? (uint32_t *)calloc ((size_t)nc_total, 4) : NULL;
			if (nc_total > 0 && (!csize || otz_deflate_chunks (ctx, job, NULL, NULL, csize, (uint32_t)nc_total, NULL) < 0)) {
				ok = 0;
			}
		}
		int any_enc = 0;
		for (zip_uint64_t k = 0; k < n_new; k++) {
			any_enc |= a->pend[idx[k]].enc != 0;
		}
		if (ok && any_enc && seal_entries (a, ctx, job, idx, n_new, out_ofs, out_size, out_total, &sealed, sofs) != 0) {
			ok = 0;
		}
		if (d_in) {
			otz_dev_free (ctx, d_in);
		}
		otz_deflate_destroy (ctx, job);
		if (!ok) {
			fprintf (stderr, "otezip-b200: GPU compress failed: %s\n", otz_last_error ());
			free (first_chunk);
			free (n_chunks);
			free (csize);
			goto done;
		}
		for (zip_uint64_t k = 0; k < n_new; k++) {
			struct otezip_entry *e = &za->entries[idx[k]];
			const uint16_t enc = a->pend[idx[k]].enc;
			e->crc32 = enc ? 0u : crc[k];   /* AE-2: no CRC of the plaintext in the clear */
			e->comp_size = out_size[k] + (enc ? AES_OVERHEAD (enc) : 0u);
			e->method = enc ? (uint16_t)METHOD_AES : method_out[k];
			a->aes[idx[k]].vendor = enc ? 2 : 0;
			a->aes[idx[k]].strength = (uint8_t)enc;
			a->aes[idx[k]].method = method_out[k];
			e->local_hdr_ofs = (uint32_t)pos;   /* (the reference gives up beyond 4 GiB, otezip.c:1140; ZIP64 here) */
			a->lfh64[idx[k]] = pos;
			/* chunk index for multi-chunk DEFLATE entries */
			uint8_t *extra = NULL;
			uint16_t extra_len = 0;
			if (enc) {
				extra_len = 11;
				extra = (uint8_t *)malloc (extra_len);
				if (!extra) {
					ok = 0;
					break;
				}
				aes_extra (extra, &a->aes[idx[k]]);
			} else if (index_enabled () && e->method == OTEZIP_METHOD_DEFLATE && n_chunks[k] >= 2 && n_chunks[k] <= OZ_EXTRA_MAX_CHUNKS) {
				extra_len = (uint16_t)(4 + 12 + 4 * n_chunks[k]);
				extra = (uint8_t *)calloc (1, extra_len);
				if (extra) {
					otezip_write_le16 (extra, OZ_EXTRA_ID);
					otezip_write_le16 (extra + 2, (uint16_t)(extra_len - 4));
					extra[4] = 1;
					otezip_write_le32 (extra + 8, chunk_bytes);
					otezip_write_le32 (extra + 12, n_chunks[k]);
					for (uint32_t c = 0; c < n_chunks[k]; c++) {
						otezip_write_le32 (extra + 16 + 4 * c, csize[first_chunk[k] + c]);
					}
				} else {
					extra_len = 0;
				}
			}
			int wrc = write_lfh (za->fp, e, extra, extra_len, streaming, enc != 0);
			free (extra);
			const uint8_t *payload = enc ? sealed + sofs[k] : out + out_ofs[k];
			if (wrc != 0 || (e->comp_size && fwrite (payload, 1, e->comp_size, za->fp) != e->comp_size) ||
				(streaming && write_descriptor (za->fp, e) != 0)) {
				ok = 0;
				break;
			}
			pos += 30 + strlen (e->name) + extra_len + e->comp_size + (streaming ? 16u : 0u);
		}
		free (first_chunk);
		free (n_chunks);
		free (csize);
		if (!ok) {
			goto done;
		}
	}
	{
		uint64_t cd_size = 0;
		for (zip_uint64_t i = 0; i < za->n_entries; i++) {
			cd_size += write_cdh (za->fp, &za->entries[i], entry_lfh (za, i), streaming && (!a->n_existing || i >= a->n_existing || (a->pend && a->pend[i].dirty)),
				aes_of (a, i));
		}
		/* otezip.c:1561-1590 truncates the counts to 16 bits and fails beyond 4 GiB (:1264); here the ZIP64 record and
		 * locator (APPNOTE 4.3.14-4.3.15) are written whenever a field does not fit */
		const int z64 = za->n_entries >= 0xFFFFu || pos >= 0xFFFFFFFFULL || cd_size >= 0xFFFFFFFFULL;
		if (z64) {
			uint8_t r[56 + 20];
			memset (r, 0, sizeof (r));
			otezip_write_le32 (r, SIG_EOCD64);
			otezip_write_le32 (r + 4, 44);          /* size of the record after this field (low word) */
			otezip_write_le16 (r + 12, 0x031e);
			otezip_write_le16 (r + 14, 45);
			otezip_write_le32 (r + 24, (uint32_t)za->n_entries);
			otezip_write_le32 (r + 28, (uint32_t)(za->n_entries >> 32));
			otezip_write_le32 (r + 32, (uint32_t)za->n_entries);
			otezip_write_le32 (r + 36, (uint32_t)(za->n_entries >> 32));
			otezip_write_le32 (r + 40, (uint32_t)cd_size);
			otezip_write_le32 (r + 44, (uint32_t)(cd_size >> 32));
			otezip_write_le32 (r + 48, (uint32_t)pos);
			otezip_write_le32 (r + 52, (uint32_t)(pos >> 32));
			const uint64_t rpos = pos + cd_size;
			otezip_write_le32 (r + 56, SIG_EOCD64_LOC);
			otezip_write_le32 (r + 56 + 8, (uint32_t)rpos);
			otezip_write_le32 (r + 56 + 12, (uint32_t)(rpos >> 32));
			otezip_write_le32 (r + 56 + 16, 1);
			if (fwrite (r, 1, sizeof (r), za->fp) != sizeof (r)) {
				goto done;
			}
		}
		uint8_t eocd[22];
		memset (eocd, 0, sizeof (eocd));
		otezip_write_le32 (eocd, SIG_EOCD);
		otezip_write_le16 (eocd + 8, za->n_entries >= 0xFFFFu ? 0xFFFFu : (uint16_t)za->n_entries);
		otezip_write_le16 (eocd + 10, za->n_entries >= 0xFFFFu ? 0xFFFFu : (uint16_t)za->n_entries);
		otezip_write_le32 (eocd + 12, cd_size >= 0xFFFFFFFFULL ? 0xFFFFFFFFu : (uint32_t)cd_size);
		otezip_write_le32 (eocd + 16, pos >= 0xFFFFFFFFULL ? 0xFFFFFFFFu : (uint32_t)pos);
		if (fwrite (eocd, 1, 22, za->fp) != 22) {
			goto done;
		}
		fflush (za->fp);
		if (a->n_existing) {
			long end = ftell (za->fp);
			if (end > 0 && ftruncate (fileno (za->fp), end) != 0) {
				goto done;
			}
		}
		rc = 0;
	}
done:
	free (idx);
	if (in) {
		otz_host_free (in);
	}
	if (out) {
		otz_host_free (out);
	}
	free (in_ofs);
	free (out_ofs);
	free (in_len);
	free (out_size);
	free (crc);
	free (method);
	free (method_out);
	free (sofs);
	if (sealed) {
		otz_host_free (sealed);
	}
	return rc;
}

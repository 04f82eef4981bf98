/* otz_gpu.h — C-ABI seam between the plain-C otezip host library and the
 * sm_100a CUDA kernels (libotezip_b200.so).  Plain pointers and sizes only.
 *
 * What each entry point replaces in the reference (paths relative to
 * /root/reference; the reference has no FFI — its "operators" are the
 * z_stream one-shot calls made from src/lib/otezip.c):
 *
 *   otz_extract_*   the per-entry body of otezip_extract_entry,
 *                   src/lib/otezip.c:399-684, for a whole batch of entries:
 *                     LFH resolve + bounds + zip-bomb guard   otezip.c:403-462
 *                     STORE                                    otezip.c:481-487
 *                     inflateInit2/inflate/inflateEnd          otezip.c:503-529
 *                                                              (src/lib/deflate-dec.inc.c:452-843)
 *                     zstdDecompressInit/zstdDecompress/End    otezip.c:542-555
 *                                                              (src/lib/zstd.inc.c:439-727)
 *                     otezip_crc32 + verdict                   otezip.c:667-679
 *                                                              (src/lib/crc32.inc.c:40-47)
 *   otz_deflate_*   otezip_compress_data's STORE/DEFLATE arms + the CRC of
 *                   zip_file_add, src/lib/otezip.c:788-852, :1124
 *                   (src/lib/deflate-enc.inc.c:199-541), for a batch of sources.
 *
 * The entry table (otz_entry[]) is what the central-directory walk
 * (otezip.c:275-396) now emits next to struct otezip_entry[].
 *
 * No CPU fallback exists behind these calls: without a CUDA device every
 * function returns OTZ_ERR_CUDA.
 */
#ifndef OTZ_GPU_H
#define OTZ_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- library return codes ---- */
#define OTZ_SUCCESS 0
#define OTZ_ERR_CUDA (-1)   /* CUDA runtime error / no device; see otz_last_error() */
#define OTZ_ERR_ARG (-2)
#define OTZ_ERR_NOMEM (-3)

/* ---- per-entry status word written by the kernels (int32) ----
 * low byte = result code, bits 8.. = advisory flags.  zip_fopen_index hands the
 * buffer to the caller iff code == OTZ_ST_OK, and no flag that the current
 * policy treats as fatal is set (see otz_status_accepts()). */
#define OTZ_ST_OK 0
#define OTZ_ST_LFH_RANGE 1     /* local_hdr_ofs / 30-byte LFH outside the image   otezip.c:411-420 */
#define OTZ_ST_LFH_SIG 2       /* LFH signature mismatch                          otezip.c:421-423 */
#define OTZ_ST_DATA_RANGE 3    /* payload outside the image                       otezip.c:438-446 */
#define OTZ_ST_ZIPBOMB 4       /* uncomp > comp*ratio+slack                       otezip.c:454-462 */
#define OTZ_ST_METHOD 5        /* method not on the GPU path (only 0, 8, 9, 93, 95; XZ: a filter other than LZMA2) otezip.c:662-665 */
#define OTZ_ST_STORE_SIZE 6    /* STORE with comp != uncomp                       otezip.c:482-485 */
#define OTZ_ST_DATA 7          /* corrupt stream (Z_DATA_ERROR class)             dec / zstd */
#define OTZ_ST_TRUNCATED 8     /* input exhausted before the stream ended (Z_BUF_ERROR class) */
#define OTZ_ST_OVERFLOW 9      /* stream produces more than uncomp_size bytes     dec:700-703, :791-793 */
#define OTZ_ST_SIZE 10         /* method 93: total_out != uncomp_size             otezip.c:555 */
#define OTZ_ST_NOPASSWD 11     /* WinZip AES entry (method 99) and no password given                 */
#define OTZ_ST_WRONGPASSWD 12  /* password verification value does not match                         */
#define OTZ_ST_AUTH 13         /* HMAC-SHA1 authentication code does not match: the ciphertext changed */
#define OTZ_ST_PENDING 0x7F    /* never touched by a kernel (internal) */
#define OTZ_ST_CODE(s) ((s) & 0xFF)
#define OTZ_STF_CRC_MISMATCH 0x100 /* otezip.c:669: fatal only under otezip_verify_crc */
#define OTZ_STF_REF_EOB 0x200      /* valid RFC 1951 stream that the reference's inflate()
                                    * rejects with Z_BUF_ERROR (dec:811-816, SURVEY.md F1) */
#define OTZ_STF_SHORT 0x400        /* stream ended before uncomp_size; tail is zero (otezip.c:500) */

/* ---- compression methods on this path (src/include/otezip/config.h:28-35) ---- */
#define OTZ_M_STORE 0
#define OTZ_M_DEFLATE 8
/* read path only: Deflate64 (PKWARE "enhanced deflate"), decoded by k_inflate<G, W, true>.  The reference rejects the
 * method, so a stream that decodes carries OTZ_STF_REF_EOB as well (handed out only when ref_compat is 0). */
#define OTZ_M_DEFLATE64 9
#define OTZ_M_ZSTD 93
/* read path only: XZ (xz streams of one LZMA2 filter each), walked by k_xz_walk and decoded by k_lzma.  The reference rejects
 * the method, so a payload that decodes carries OTZ_STF_REF_EOB as well (handed out only when ref_compat is 0). */
#define OTZ_M_XZ 95
/* write path only: or-ed into method[i], compression level 1 ("fastest": one match candidate per position instead of the
 * eight-way search at the start of every token; about 3x the speed at 0.85x the ratio on text) */
#define OTZ_M_FAST 0x100
/* write path only: or-ed into method 8 alone (OTZ_M_DEFLATE | OTZ_M_BEST), the "best" level (libzip levels 7-9): hash
 * chains over every position of a chunk, each position searched 128 links deep, two-step lazy parse (k_deflate_best.cuh).
 * The chunk layout is that of the other levels.  otz_deflate_plan rejects it with OTZ_M_FAST, STORE or method 93. */
#define OTZ_M_BEST 0x200

/* One row of the device-side entry table (32 bytes). */
typedef struct otz_entry {
	uint64_t lfh_ofs;     /* offset of the local file header in the archive image */
	uint64_t out_ofs;     /* offset of this entry's bytes in the output arena */
	uint32_t comp_size;
	uint32_t uncomp_size;
	uint32_t crc32;       /* expected CRC-32 from the central directory */
	uint16_t method;
	uint16_t flags;       /* OTZ_EF_* */
} otz_entry;

/* Row flags.  Archives written by this library carry, in the LFH extra field of a multi-chunk DEFLATE entry,
 * the compressed size of each independently decodable chunk (otezip/zip.h, "chunk index").  The directory walk
 * then emits one PARENT row (resolved, CRC'd and reported like any entry, but not decoded as one stream) plus one
 * CHUNK row per chunk: lfh_ofs = offset of the chunk's first byte in the image, out_ofs = where its bytes go,
 * crc32 = row number of its parent.  A failing chunk fails its parent. */
#define OTZ_EF_PARENT 0x0001
#define OTZ_EF_CHUNK 0x0002
#define OTZ_EF_LAST_CHUNK 0x0004   /* must end with the stream's final block */

typedef struct otz_extract_opts {
	int ignore_zipbomb;       /* otezip_ignore_zipbomb        otezip.c:166 */
	uint64_t max_ratio;       /* otezip_max_expansion_ratio   otezip.c:164 */
	uint64_t max_slack;       /* otezip_max_expansion_slack   otezip.c:165 */
	int verify_only;          /* 1: STORE entries are CRC-checked in place and not copied to
	                           *    the arena (BASELINE configs[1] "STORE + CRC-32 verify only") */
} otz_extract_opts;

typedef struct otz_ctx otz_ctx;     /* one per (process, device): stream, tables, scratch */
typedef struct otz_plan otz_plan;   /* a resident entry table + its work lists */

/* ---- context ---- */
int otz_device_count(void);
int otz_ctx_create(int device, otz_ctx **out);
void otz_ctx_destroy(otz_ctx *ctx);
const char *otz_last_error(void);
/* Debug build only (libotezip_b200_dbg.so, -DOTZ_BOUNDS_CHECK): violations counted by the kernels' software bounds
 * checks since the library was loaded, one counter per check site; returns the number of counters, -1 when the checks
 * are not compiled in (the release library). */
int otz_debug_violations(uint64_t *out, int cap);
int otz_sm_count(otz_ctx *ctx);
int otz_pci_bus_id(otz_ctx *ctx, char *buf, int len);   /* for NVML clock sampling */

/* ---- device / pinned memory and copies (all on the context's stream) ---- */
int otz_dev_alloc(otz_ctx *ctx, uint64_t bytes, void **dptr);   /* padded by 64 bytes */
int otz_dev_free(otz_ctx *ctx, void *dptr);
int otz_host_alloc(uint64_t bytes, void **hptr);                /* pinned */
int otz_host_free(void *hptr);
int otz_h2d(otz_ctx *ctx, void *dptr, const void *hptr, uint64_t bytes);  /* async */
int otz_d2h(otz_ctx *ctx, void *hptr, const void *dptr, uint64_t bytes);  /* async */
int otz_dev_memset(otz_ctx *ctx, void *dptr, int value, uint64_t bytes);  /* async */
int otz_sync(otz_ctx *ctx);

/* ---- device timing on the launching stream (cudaEvent pair) ---- */
int otz_timer_start(otz_ctx *ctx);
int otz_timer_stop(otz_ctx *ctx, float *ms);   /* records, synchronises, returns elapsed */
/* per-phase event timing of otz_extract_run (ms).  otz_profile_enable(ctx,1) resets the run
 * counter; every later run records 5 events on the stream (no synchronisation); the last 64
 * runs can be read back by index after the timed region. */
int otz_profile_enable(otz_ctx *ctx, int on);
int otz_profile_runs(otz_ctx *ctx);
int otz_profile_get(otz_ctx *ctx, int run, float *ms_resolve, float *ms_decode, float *ms_crc, float *ms_finalize);
/* kernel launches issued by this context so far */
uint64_t otz_launch_count(otz_ctx *ctx);
/* write `bytes` of scratch larger than L2 (flushes L2 between timed iterations) */
int otz_flush_l2(otz_ctx *ctx);

/* ---- read path ---- */
/* Upload the entry table and build the work lists (host side of the CD walk). */
int otz_plan_create(otz_ctx *ctx, const otz_entry *entries, uint32_t n, const otz_extract_opts *opts,
	otz_plan **out);
void otz_plan_destroy(otz_ctx *ctx, otz_plan *plan);
/* Launch the batch on device-resident buffers (asynchronous). d_out may be NULL
 * only when every entry is STORE and opts.verify_only is set. */
int otz_extract_run(otz_ctx *ctx, otz_plan *plan, const uint8_t *d_archive, uint64_t archive_len,
	uint8_t *d_out, uint64_t out_len);
/* Copy per-entry results back (synchronises). crc = computed CRC-32 (valid when
 * the code is OTZ_ST_OK), status = status words. Either may be NULL. */
int otz_extract_results(otz_ctx *ctx, otz_plan *plan, uint32_t *crc, int32_t *status);
/* Host-buffer convenience: H2D image, run, D2H arena + results. */
int otz_extract_host(otz_ctx *ctx, const uint8_t *archive, uint64_t archive_len, const otz_entry *entries,
	uint32_t n, const otz_extract_opts *opts, uint8_t *out, uint64_t out_len, uint32_t *crc, int32_t *status);

/* ---- write path ----
 * Batched otezip_compress_data (otezip.c:788-852) + CRC (otezip.c:1124) for n sources laid out in one
 * input buffer: source i = in[in_ofs[i] .. in_ofs[i]+in_len[i]), requested method[i] in {0, 8, 93}
 * (93: real Zstandard frames, one block per 65,280-byte chunk, k_zstd_enc.cuh — an extension: the reference's method-93
 * writer is a stub that always ends up at STORE).
 * Per source: zero length -> STORE; DEFLATE whose stream is not smaller than the input -> STORE
 * (otezip.c:793-801, :846-850).  Results: method_out[i], out_size[i], out_ofs[i] (offset in the dense
 * output arena), crc[i] = CRC-32 of the uncompressed bytes. */
typedef struct otz_deflate_job otz_deflate_job;
int otz_deflate_plan(otz_ctx *ctx, const uint64_t *in_ofs, const uint32_t *in_len, const uint16_t *method, uint32_t n,
	otz_deflate_job **out);
void otz_deflate_destroy(otz_ctx *ctx, otz_deflate_job *job);
/* Launch CRC + compress + compaction on a device-resident input (asynchronous). */
int otz_deflate_run(otz_ctx *ctx, otz_deflate_job *job, const uint8_t *d_in, uint64_t in_bytes);
/* Per-source results (synchronises; any pointer may be NULL). *total = bytes in the dense arena. */
int otz_deflate_results(otz_ctx *ctx, otz_deflate_job *job, uint64_t *out_ofs, uint32_t *out_size, uint32_t *crc,
	uint16_t *method_out, uint64_t *total);
/* Chunk layout of the job: first_chunk[i] / n_chunks[i] per source, csize[] = compressed bytes of every chunk
 * (valid after otz_deflate_results; the bytes of a DEFLATE source are its chunks back to back, each one
 * independently decodable).  chunk_bytes = uncompressed bytes per chunk.  Returns the total number of chunks. */
int otz_deflate_chunks(otz_ctx *ctx, otz_deflate_job *job, uint32_t *first_chunk, uint32_t *n_chunks, uint32_t *csize,
	uint32_t csize_cap, uint32_t *chunk_bytes);
/* Device pointer of the dense output arena (valid until the job is destroyed). */
const uint8_t *otz_deflate_device_output(otz_deflate_job *job);
/* Copy the dense arena (first `bytes` bytes) to the host (synchronises). */
int otz_deflate_fetch(otz_ctx *ctx, otz_deflate_job *job, uint8_t *out, uint64_t bytes);
/* Host-buffer convenience: H2D input, run, D2H results + arena.  out_cap >= sum(in_len) always suffices. */
int otz_deflate_host(otz_ctx *ctx, const uint8_t *in, uint64_t in_bytes, const uint64_t *in_ofs, const uint32_t *in_len,
	const uint16_t *method, uint32_t n, uint8_t *out, uint64_t out_cap, uint64_t *out_ofs, uint32_t *out_size,
	uint32_t *crc, uint16_t *method_out, uint64_t *total);

/* Same, plus produced[i] = bytes the stream of entry i actually produced (== uncomp_size except for DEFLATE
 * streams that end early, whose tail is zero: OTZ_STF_SHORT). */
int otz_extract_host_ex(otz_ctx *ctx, const uint8_t *archive, uint64_t archive_len, const otz_entry *entries,
	uint32_t n, const otz_extract_opts *opts, uint8_t *out, uint64_t out_len, uint32_t *crc, int32_t *status,
	uint32_t *produced);
int otz_extract_produced(otz_ctx *ctx, otz_plan *plan, uint32_t *produced);

/* DEFLATE streams of the run last collected with otz_extract_results that the lane-per-stream decoder
 * (k_inflate_tok/k_inflate_lz) declined and the warp-per-stream decoder (k_inflate) decoded instead:
 * error and short streams, stored blocks with payload, code sets beyond the fixed table budget.  Both decoders
 * implement dec:547-831 with identical results; this is a performance counter.  Deflate64 streams always run on
 * k_inflate and are not counted. */
uint32_t otz_inflate_fallbacks(otz_ctx *ctx);

/* ---- multi-GPU sharding (SURVEY.md §8e; the reference has no counterpart: entries are independent,
 * otezip.c:399-477) ----
 * Split entries [0, n) into `parts` contiguous index ranges balanced by comp_size + uncomp_size (what a device
 * reads and writes): first[g] .. first[g + 1] is the range of part g, first[parts] = n.  Contiguous ranges keep
 * each part a contiguous byte range of the archive.  Pure host code (no device needed). */
int otz_partition(const otz_entry *entries, uint32_t n, uint32_t parts, uint32_t *first);
/* otz_extract_host_ex over several devices of one box: one context per device, the table cut by otz_partition, every
 * device handed only its byte range of the image and of the arena, one host thread per device, no collective.
 * Results are identical to the single-device call. */
int otz_extract_host_multi(otz_ctx *const *ctxs, uint32_t n_ctx, const uint8_t *archive, uint64_t archive_len,
	const otz_entry *entries, uint32_t n, const otz_extract_opts *opts, uint8_t *out, uint64_t out_len, uint32_t *crc,
	int32_t *status, uint32_t *produced);

/* ---- WinZip AES (AE-1 / AE-2, method 99; k_aes.cuh) ----
 * An encrypted payload is  salt (8/12/16 bytes for strength 1/2/3 = AES-128/192/256) | verification value (2) | ciphertext |
 * authentication code (10).  Keys: PBKDF2-HMAC-SHA1(password, salt, 1000 iterations, 2*keylen + 2) = AES key | HMAC key |
 * verification value.  Cipher: AES-CTR, little-endian counter from 1.  Code: HMAC-SHA1 over the ciphertext, first 10 bytes. */
#define OTZ_AES_NOPASSWORD 0xFFFFu
typedef struct otz_aes_entry {
	uint64_t payload_ofs;   /* open: the payload in d_src;  seal: where the payload goes in d_out */
	uint64_t data_ofs;      /* open: where the synthetic 30-byte local header goes in d_plain (the plaintext follows it);
	                         * seal: the bytes to encrypt in d_in */
	uint32_t size;          /* open: payload bytes (the directory's compressed size);  seal: bytes to encrypt */
	uint16_t strength;      /* 1 / 2 / 3 */
	uint16_t password;      /* index into passwords[]; OTZ_AES_NOPASSWORD = none (open reports OTZ_ST_NOPASSWD) */
} otz_aes_entry;
/* Decrypt n entries of d_src into the plaintext image d_plain (asynchronous): key derivation, then AES-CTR on the context's
 * stream, the authentication codes on a side stream next to it.  Each entry of the image is a local header (signature, every
 * other field zero) followed by the decrypted payload, so otz_plan_create / otz_extract_run decode the image as an archive.
 * passwords[] are NUL-terminated byte strings.  d_src must stay valid until otz_aes_status. */
int otz_aes_open(otz_ctx *ctx, const uint8_t *d_src, uint64_t src_len, const otz_aes_entry *ents, uint32_t n,
	const char *const *passwords, uint32_t n_pw, uint8_t *d_plain, uint64_t plain_len);
/* Join the side stream, clear the device key scratch and return the verdict of each entry of the last otz_aes_open
 * (synchronises): OTZ_ST_OK, OTZ_ST_NOPASSWD, OTZ_ST_WRONGPASSWD or OTZ_ST_AUTH. */
int otz_aes_status(otz_ctx *ctx, int32_t *status);
/* Device time of the phases of the last otz_aes_open (valid after otz_aes_status), ms; any pointer may be NULL.  The
 * authentication codes run beside the decryption: ms_mac counts from the end of the key derivation. */
int otz_aes_times(otz_ctx *ctx, float *ms_kdf, float *ms_ctr, float *ms_mac);
/* Encrypt n entries of d_in (e.g. otz_deflate_device_output) into d_out as salt | verification value | ciphertext | code,
 * salts[16 * i ..] supplying the salt of entry i (its first 8/12/16 bytes).  Synchronises; the key scratch is cleared. */
int otz_aes_seal(otz_ctx *ctx, const uint8_t *d_in, uint64_t in_len, const otz_aes_entry *ents, uint32_t n, const uint8_t *salts,
	const char *const *passwords, uint32_t n_pw, uint8_t *d_out, uint64_t out_len);

/* Policy helper shared by the host library and the tests: does a status word
 * mean "zip_fopen_index returns the buffer" under the given globals?
 * ref_compat != 0 reproduces the reference's end-of-block rule (F1). */
int otz_status_accepts(int32_t status, int verify_crc, int ref_compat);

#ifdef __cplusplus
}
#endif
#endif

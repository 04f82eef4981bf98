/* otezip/zip.h — the libzip-subset API of otezip, as exported by libotezip_b200.so.
 *
 * This header is the drop-in boundary: every type, field order, constant and prototype below has the
 * layout of the reference's src/include/otezip/zip.h (structs :78-110, flags :130-143, errors :153-161,
 * zip_stat :173-182, prototypes :192-215, globals :222-231), because callers such as the otezip CLI
 * reach into the structs (za->entries[i].name, za->default_method, zf->data / zf->size).
 *
 * What differs is behind it: zip_fopen_index() decodes entries in batches on the GPU (the first call
 * for an entry triggers a batch that covers its neighbours), and zip_file_add() only queues the source;
 * compression, CRC and all writes happen in zip_close() as one GPU batch, so
 * zip_set_file_compression() after zip_file_add() takes effect (libzip semantics).
 */
#ifndef OTEZIP_H_
#define OTEZIP_H_

#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "config.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef uint64_t zip_uint64_t;
typedef int64_t zip_int64_t;
typedef int zip_flags_t;
typedef int32_t zip_int32_t;
typedef uint32_t zip_uint32_t;
typedef uint16_t zip_uint16_t;
typedef uint8_t zip_uint8_t;

/* ---- records (field order is ABI) ---- */
struct otezip_entry {
	char *name;
	uint32_t local_hdr_ofs;
	uint32_t comp_size;
	uint32_t uncomp_size;
	uint16_t method;
	uint32_t crc32;
	uint16_t file_time;
	uint16_t file_date;
	uint32_t external_attr;
};

struct zip {
	FILE *fp;
	struct otezip_entry *entries;
	zip_uint64_t n_entries;
	int mode;                 /* 0 read, 1 write */
	zip_uint64_t next_index;
	uint16_t default_method;  /* method given to entries added from now on */
};

struct zip_file {
	uint8_t *data;            /* whole uncompressed entry; owned by the library */
	uint32_t size;
	zip_uint64_t pos;
};

struct zip_source {
	const void *buf;
	zip_uint64_t len;
	int freep;
};

struct otezip_error {
	int zip_err;
	int sys_err;
};

struct zip_stat {
	zip_uint64_t valid;
	const char *name;
	zip_uint64_t index;
	zip_uint64_t size;
	zip_uint64_t comp_size;
	time_t mtime;
	zip_uint32_t crc;
	zip_uint16_t comp_method;
};

typedef struct zip zip_t;
typedef struct zip_file zip_file_t;
typedef struct zip_source zip_source_t;
typedef struct otezip_error zip_error_t;
typedef struct zip_stat zip_stat_t;
typedef struct zip otezip_archive;
typedef struct zip_file otezip_file;
typedef struct zip_source otezip_src_buf;

/* ---- constants ---- */
#define ZIP_RDONLY 0
#define ZIP_CREATE 1
#define ZIP_EXCL 2
#define ZIP_TRUNCATE 8

#define ZIP_CM_STORE 0
#define ZIP_CM_DEFLATE 8
/* Deflate64 (PKWARE "enhanced deflate"; 7-Zip -mm=Deflate64, Windows' zipped folders for large inputs): read only.  The
 * reference rejects the method, so with the default otezip_ref_compat = 1 zip_fopen_index returns NULL for such an entry
 * (otezip_b200_entry_status: OTZ_ST_OK | OTZ_STF_REF_EOB when its stream is valid); with 0 it hands out the bytes. */
#define ZIP_CM_DEFLATE64 9
/* XZ (xz streams with one LZMA2 filter; libzip ZIP_CM_XZ, 7-Zip -mm=xz): read only, under the same rule as Deflate64 --
 * with otezip_ref_compat = 1 zip_fopen_index returns NULL for such an entry (otezip_b200_entry_status: OTZ_ST_OK |
 * OTZ_STF_REF_EOB when its payload is valid); with 0 it hands out the bytes.  Filters other than LZMA2 (BCJ, delta) give
 * OTZ_ST_METHOD. */
#define ZIP_CM_XZ 95

#define ZIP_UINT64_MAX ((zip_uint64_t)-1)

#define ZIP_ER_OK 0
#define ZIP_ER_READ 5
#define ZIP_ER_NOENT 9
#define ZIP_ER_EXISTS 10
#define ZIP_ER_OPEN 11
#define ZIP_ER_INVAL 18
#define ZIP_ER_NOZIP 19
#define ZIP_ER_INCONS 21
#define ZIP_ER_RDONLY 25
/* libzip's encryption error codes, for callers that use the names.  This subset has no per-archive error state: the
 * calls fail with NULL / -1, and the reason an encrypted entry did not open is its status word
 * (otezip_b200_entry_status: OTZ_ST_NOPASSWD, OTZ_ST_WRONGPASSWD, OTZ_ST_AUTH of include/otz_gpu.h). */
#define ZIP_ER_ENCRNOTSUPP 24
#define ZIP_ER_NOPASSWD 26
#define ZIP_ER_WRONGPASSWD 27

/* encryption methods (libzip values); only WinZip AES is implemented, traditional PKWARE encryption is not */
#define ZIP_EM_NONE 0
#define ZIP_EM_TRAD_PKWARE 1
#define ZIP_EM_AES_128 0x0101
#define ZIP_EM_AES_192 0x0102
#define ZIP_EM_AES_256 0x0103

#define ZIP_STAT_NAME 0x0001u
#define ZIP_STAT_INDEX 0x0002u
#define ZIP_STAT_SIZE 0x0004u
#define ZIP_STAT_COMP_SIZE 0x0008u
#define ZIP_STAT_MTIME 0x0010u
#define ZIP_STAT_CRC 0x0020u
#define ZIP_STAT_COMP_METHOD 0x0040u

/* ---- little-endian field helpers (static inline, usable from any unit) ---- */
static inline uint16_t otezip_read_le16(const uint8_t *p) { return (uint16_t)(p[0] | (p[1] << 8)); }
static inline uint32_t otezip_read_le32(const uint8_t *p) {
	return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
static inline uint64_t otezip_read_le64(const uint8_t *p) {
	return (uint64_t)otezip_read_le32(p) | ((uint64_t)otezip_read_le32(p + 4) << 32);
}
static inline void otezip_write_le16(uint8_t *p, uint16_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }
static inline void otezip_write_le32(uint8_t *p, uint32_t v) {
	otezip_write_le16(p, (uint16_t)v);
	otezip_write_le16(p + 2, (uint16_t)(v >> 16));
}
static inline void otezip_write_le64(uint8_t *p, uint64_t v) {
	otezip_write_le32(p, (uint32_t)v);
	otezip_write_le32(p + 4, (uint32_t)(v >> 32));
}

/* ---- archive lifecycle and read path ---- */
zip_t *zip_open(const char *path, int flags, int *errorp);
zip_t *zip_open_from_source(zip_source_t *src, int flags, zip_error_t *error);
int zip_close(zip_t *za);
zip_uint64_t zip_get_num_files(zip_t *za);
zip_int64_t zip_name_locate(zip_t *za, const char *fname, zip_flags_t flags);
const char *zip_get_name(zip_t *za, zip_uint64_t index, zip_flags_t flags);
zip_file_t *zip_fopen_index(zip_t *za, zip_uint64_t index, zip_flags_t flags);
int zip_fclose(zip_file_t *zf);
zip_int64_t zip_fread(zip_file_t *zf, void *buf, zip_uint64_t nbytes);
int zip_stat(zip_t *za, const char *fname, zip_flags_t flags, zip_stat_t *st);
int zip_stat_index(zip_t *za, zip_uint64_t index, zip_flags_t flags, zip_stat_t *st);
void zip_stat_init(zip_stat_t *st);

/* ---- write path ---- */
zip_source_t *zip_source_buffer(zip_t *za, const void *data, zip_uint64_t len, int freep);
zip_source_t *zip_source_buffer_create(const void *data, zip_uint64_t len, int freep, zip_error_t *error);
void zip_source_free(zip_source_t *src);
zip_int64_t zip_file_add(zip_t *za, const char *name, zip_source_t *src, zip_flags_t flags);
zip_int64_t zip_add(zip_t *za, const char *name, zip_source_t *src);
int zip_file_replace(zip_t *za, zip_uint64_t index, zip_source_t *src, zip_flags_t flags);
int zip_replace(zip_t *za, zip_uint64_t index, zip_source_t *src);
/* comp_flags is the compression level, as in libzip: 0 = default, 1-3 = fast (one match candidate per position),
 * 4-6 = default (eight-way search at token starts), 7-9 = best (DEFLATE only: hash chains searched at every position,
 * about the ratio of zlib's level 9 on independent 64 KiB chunks).  Every level writes the same independently decodable
 * chunks.  Method 93 takes 1-3 as fast and every other level as its default. */
int zip_set_file_compression(zip_t *za, zip_uint64_t index, zip_int32_t comp, zip_uint32_t comp_flags);

int otezip_method_from_string(const char *method_name);

/* ---- WinZip AES encryption (method 99, AE-1 / AE-2; libzip's calls) ----
 * Reading: an entry whose directory method is 99 is decrypted with the archive's default password (zip_fopen_index) or the
 * one given (zip_fopen_index_encrypted), then decoded like any entry of its actual method; zip_stat keeps reporting 99.  A
 * missing password, a wrong one and a failed authentication code make the open fail (otezip_b200_entry_status tells which:
 * OTZ_ST_NOPASSWD, OTZ_ST_WRONGPASSWD, OTZ_ST_AUTH); no byte of an entry whose code does not match is ever handed out.
 * Writing: zip_file_set_encryption on an entry added or replaced in this session makes zip_close write it as AE-2 (CRC field
 * 0, the code is the integrity check) with a fresh random salt.  Passwords are wiped from the library's memory on zip_close. */
int zip_set_default_password(zip_t *za, const char *password);   /* NULL clears it */
zip_file_t *zip_fopen_index_encrypted(zip_t *za, zip_uint64_t index, zip_flags_t flags, const char *password);
int zip_file_set_encryption(zip_t *za, zip_uint64_t index, zip_uint16_t method, const char *password);   /* NULL: the default */
int zip_encryption_method_supported(zip_uint16_t method, int encode);
/* libzip: 1 when entries of this compression method can be read (compress == 0: 0, 8, 9, 93, 95) or written (compress != 0:
 * 0, 8, 93) */
int zip_compression_method_supported(zip_int32_t method, int compress);

/* ---- B200 build additions (not in the reference) ---- */
/* Emit the device-side entry table of an archive opened for reading: n rows of struct otz_entry
 * (include/otz_gpu.h) with out_ofs laid out as 16-byte aligned prefix sums.  Returns rows written. */
zip_uint64_t otezip_b200_entry_table(zip_t *za, void *otz_entries, zip_uint64_t max_rows);
/* Raw status word (OTZ_ST_* | OTZ_STF_*) of the last attempt to extract entry `index`, or -1. */
int otezip_b200_entry_status(zip_t *za, zip_uint64_t index);

#ifdef __cplusplus
}
#endif

/* ---- runtime switches (same names and defaults as the reference, otezip.c:157-166) ---- */
extern int otezip_verify_crc;                 /* 1: CRC mismatch makes zip_fopen_index fail */
extern uint64_t otezip_max_expansion_ratio;   /* zip-bomb guard: uncomp <= comp*ratio + slack */
extern uint64_t otezip_max_expansion_slack;
extern int otezip_ignore_zipbomb;
/* B200 build: 1 (default) reproduces the reference inflater's end-of-input rule (SURVEY.md F1) so that
 * accept/reject is bit-identical; 0 accepts every valid RFC 1951 stream, and Deflate64 and XZ entries.  The environment variable
 * OTEZIP_REF_COMPAT=0 sets the initial value (read when the library is loaded). */
extern int otezip_ref_compat;
/* Extension (SURVEY.md §8f rank 2): 1 = zip_close writes every entry in the STREAMING layout — general-purpose flag
 * bit 3, CRC and sizes zero in the local header and a data descriptor (PK\7\8, CRC-32, sizes) behind the payload —
 * what a writer to a non-seekable sink has to emit.  The reference's reader tolerates bit 3 (it takes CRC and sizes
 * from the central directory, otezip.c:355-358, :371-377), and so does this one.  Default 0: the reference's layout.
 * Also set by the environment variable OTEZIP_DATA_DESCRIPTORS=1. */
extern int otezip_write_data_descriptors;
/* Extension (SURVEY.md §8f rank 3): 1 = method 93 means REAL Zstandard (RFC 8878) frames on both paths: zip_close
 * compresses entries set to ZIP_CM_ZSTD / `-z zstd` with the GPU Zstandard encoder (the reference's raw-block stub always
 * ends up at STORE, otezip.c:894-899), and zip_fopen_index hands out real frames, which the reference's reader rejects
 * (SURVEY F3).  Default 0: the reference's observable behaviour.  Also set by OTEZIP_ZSTD_FRAMES=1. */
extern int otezip_zstd_frames;

#endif /* OTEZIP_H_ */

/* otezip/config.h — build switches and method ids of the B200 build.
 * Same macro names and values as the reference's src/include/otezip/config.h:6-35 (the method ids are
 * the ZIP APPNOTE numbers and part of the on-disk format); methods 0, 8 and 93 are implemented by the GPU path, which also
 * reads 9 (Deflate64) and 95 (XZ, otz_gpu.h: OTZ_M_XZ); the rest are reported as unsupported (OTZ_ST_METHOD). */
#ifndef OTEZIP_CONFIG_H
#define OTEZIP_CONFIG_H

#define OTEZIP_VERSION_MAJOR 0
#define OTEZIP_VERSION_MINOR 4
#define OTEZIP_VERSION_PATCH 8
#define OTEZIP_STR2(x) #x
#define OTEZIP_STR(x) OTEZIP_STR2(x)
#define OTEZIP_VERSION OTEZIP_STR(OTEZIP_VERSION_MAJOR) "." OTEZIP_STR(OTEZIP_VERSION_MINOR) "." OTEZIP_STR(OTEZIP_VERSION_PATCH)
#define OTEZIP_B200 1

#define OTEZIP_ENABLE_STORE 1
#define OTEZIP_ENABLE_DEFLATE 1
#define OTEZIP_ENABLE_ZSTD 1

enum {
	OTEZIP_METHOD_STORE = 0,
	OTEZIP_METHOD_DEFLATE = 8,
	OTEZIP_METHOD_LZMA = 14,
	OTEZIP_METHOD_ZSTD = 93,
	OTEZIP_METHOD_LZ4 = 94,
	OTEZIP_METHOD_BROTLI = 97,
	OTEZIP_METHOD_LZFSE = 100
};

#endif

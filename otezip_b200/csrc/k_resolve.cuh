// k_resolve.cuh — per-entry local-header resolve, bounds and zip-bomb guard.
//
// Replaces the head of otezip_extract_entry (/root/reference/src/lib/otezip.c:399-487):
// one thread per row of the device entry table reads the 30-byte LFH straight
// from the archive image in HBM and decides accept/reject exactly as the
// reference does before it touches a codec.
#pragma once
#include "otz_common.cuh"

__global__ void k_resolve(const uint8_t *__restrict__ archive, uint64_t archive_len, uint64_t out_len,
	const otz_entry *__restrict__ ents, uint32_t n, OtzEntryState *__restrict__ est, int32_t *__restrict__ status,
	uint32_t *__restrict__ acc, uint32_t *__restrict__ produced, otz_extract_opts opts) {
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) {
		return;
	}
	const otz_entry e = ents[i];
	acc[i] = 0;
	produced[i] = e.uncomp_size;   // DEFLATE streams that end early overwrite this (zero-padded tail)
	est[i].data_ofs = 0;
	int32_t st = OTZ_ST_OK;
	if (e.flags & OTZ_EF_CHUNK) {
		// a chunk of an indexed DEFLATE entry: lfh_ofs is the payload offset itself
		if (e.method != OTZ_M_DEFLATE || e.lfh_ofs > archive_len || archive_len - e.lfh_ofs < e.comp_size || e.out_ofs > out_len ||
			out_len - e.out_ofs < e.uncomp_size) {
			st = OTZ_ST_DATA_RANGE;
		}
		est[i].data_ofs = e.lfh_ofs;
		status[i] = st;
		return;
	}
	do {
		// otezip.c:411-420: seek to the LFH and read 30 bytes
		if (e.lfh_ofs > archive_len || archive_len - e.lfh_ofs < 30) {
			st = OTZ_ST_LFH_RANGE;
			break;
		}
		const uint8_t *lfh = archive + e.lfh_ofs;
		if (ld_le32(lfh) != OTZ_SIG_LFH) {  // otezip.c:421-423
			st = OTZ_ST_LFH_SIG;
			break;
		}
		// otezip.c:429-446
		uint64_t data_ofs = e.lfh_ofs + 30ull + ld_le16(lfh + 26) + ld_le16(lfh + 28);
		if (data_ofs > archive_len || (uint64_t)e.comp_size > OTZ_MAX_PAYLOAD || (uint64_t)e.uncomp_size > OTZ_MAX_PAYLOAD ||
			data_ofs + e.comp_size > archive_len) {
			st = OTZ_ST_DATA_RANGE;
			break;
		}
		est[i].data_ofs = data_ofs;
		// otezip.c:454-462
		if (!opts.ignore_zipbomb && e.comp_size > 0) {
			uint64_t allowed = (uint64_t)e.comp_size * opts.max_ratio + opts.max_slack;
			if ((uint64_t)e.uncomp_size > allowed) {
				st = OTZ_ST_ZIPBOMB;
				break;
			}
		}
		if (e.method == OTZ_M_STORE) {  // otezip.c:481-485
			if (e.comp_size != e.uncomp_size) {
				st = OTZ_ST_STORE_SIZE;
				break;
			}
		} else if (e.method != OTZ_M_DEFLATE && e.method != OTZ_M_DEFLATE64 && e.method != OTZ_M_ZSTD && e.method != OTZ_M_XZ) {  // otezip.c:662-665
			st = OTZ_ST_METHOD;
			break;
		}
		// the arena slice must exist unless this entry is verified in place
		bool in_place = opts.verify_only && e.method == OTZ_M_STORE;
		if (!in_place && (e.out_ofs > out_len || out_len - e.out_ofs < e.uncomp_size)) {
			st = OTZ_ST_DATA_RANGE;
			break;
		}
	} while (0);
	status[i] = st;
}

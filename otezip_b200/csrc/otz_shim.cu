// otz_shim.cu — the extern "C" seam declared in include/otz_gpu.h: device/stream management,
// H2D/D2H, work-list construction and kernel launches.  CUDA runtime only; no torch, no NCCL.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "k_copy.cuh"
#include "k_crc32.cuh"
#include <string>
#include <thread>
#include "k_inflate.cuh"
#include "k_inflate2.cuh"
#include "k_inflate3.cuh"
#include "k_deflate.cuh"
#include "k_deflate_best.cuh"
#include "k_resolve.cuh"
#include "k_zstd_tok.cuh"
#include "k_aes.cuh"
#include "k_xz.cuh"
#include "otz_common.cuh"

static thread_local char g_err[512] = "";

static int fail_cuda(cudaError_t e, const char *what, int line = 0) {
	snprintf(g_err, sizeof(g_err), "%s (otz_shim.cu:%d): %s", what, line, cudaGetErrorString(e));
	return OTZ_ERR_CUDA;
}
#define CK(call)                                    \
	do {                                            \
		cudaError_t e_ = (call);                    \
		if (e_ != cudaSuccess) {                    \
			return fail_cuda(e_, #call, __LINE__);  \
		}                                           \
	} while (0)

// ring of the LZ executor for huge (segmented) streams: few streams, each one the critical path — a large ring keeps
// most match sources in shared memory
#define OTZ_SEG_RING 16384
#define OTZ_PROF_SLOTS 64
struct otz_ctx {
	int device;
	int sm_count;
	cudaStream_t stream, stream2, stream3, stream4;
	cudaEvent_t ev0, ev1, ev_fork, ev_join, ev_join3, ev_join4;
	cudaEvent_t pev[OTZ_PROF_SLOTS][5];
	int profile;
	uint32_t prof_runs;      // runs recorded since otz_profile_enable(ctx, 1)
	void *d_arch_cache, *d_out_cache;   // grow-only device buffers behind otz_extract_host
	uint64_t arch_cache_bytes, out_cache_bytes;
	OtzCrcTables *d_tabs;
	uint8_t *d_flush;
	uint64_t flush_bytes;
	uint64_t launches;
	int inflate_tile;   // lanes per DEFLATE stream (OTZ_INFLATE_TILE; 0 = per batch)
	int inflate_ring;   // bytes of shared-memory output ring per stream (OTZ_INFLATE_RING; 0 = per batch)
	int inflate_mode;   // OTZ_INFLATE_MODE: 0 = two-phase (k_inflate_spec + k_inflate_lz, k_inflate as fallback), 1 ("legacy") = k_inflate only
	int lz_ring;        // OTZ_LZ_RING: ring bytes per warp of k_inflate_lz (4096 / 8192 / 16384)
	uint32_t last_fallbacks;   // DEFLATE streams of the last collected run that phase A handed to k_inflate
	int huge_legacy;        // OTZ_HUGE_MODE=legacy: huge DEFLATE entries on k_inflate<32,16384> instead of the segmented decode
	uint8_t *d_ztok_cache;  // grow-only token scratch of the two-phase Zstandard path
	uint64_t ztok_cache_bytes;
	uint8_t *d_spec_tmp;    // temp token slots of k_inflate_spec: 4 regions (regular streams + three size groups of huge ones) of one slot per resident lane
	uint64_t spec_tmp_region;
	uint8_t *d_tok_cache;   // grow-only token scratch of the two-phase inflate (literals + sequence records)
	uint64_t tok_cache_bytes;
	int seg_serial;         // OTZ_SEG_EXEC=serial: one warp walks the chain of a huge stream (no parallel segment execution)
	int seg_ring;           // OTZ_SEG_PAR_RING: ring elements per warp of the parallel segment executor (4096 / 8192)
	uint16_t *d_sym_cache;  // grow-only symbol buffer of the parallel segment execution
	uint64_t sym_cache_elems;
	otz_ctx *pipe[2];       // child contexts (own streams and scratch) of the pipelined host call otz_extract_host
	std::vector<otz_plan *> pc_plans;   // sub-plans of the last pipelined call (reused when the same table comes again)
	std::vector<otz_entry> pc_ents;
	otz_extract_opts pc_opts;
	uint32_t pc_n;
	void *h_res;            // pinned staging of its per-entry results
	uint64_t h_res_bytes;
	uint64_t sym_limit;     // OTZ_SEG_SYM_LIMIT: cap of the symbol buffer in elements (tests: streams that do not fit are walked by one warp)
	struct OtzAesRun *aes;  // device state of the last otz_aes_open / otz_aes_seal (created on first use)
	cudaStream_t stream_d64[2];   // Deflate64 entries (large / small), beside the DEFLATE work of the same run
	cudaEvent_t ev_d64_fork, ev_d64_join[2];
	cudaStream_t stream_xz;       // XZ entries: walk, decode, verdicts, beside the other work of the same run
	cudaEvent_t ev_xz_fork, ev_xz_join;
};

struct otz_plan {
	uint32_t n;
	otz_extract_opts opts;
	otz_entry *d_ents;
	OtzEntryState *d_est;
	int32_t *d_status;
	uint32_t *d_acc, *d_crc, *d_produced;
	OtzCrcChunk *d_chunks;
	uint32_t n_chunks;
	uint32_t n_store_chunks;   // chunks [0, n_store_chunks) belong to STORE entries
	uint32_t *d_inflate_list, n_inflate;   // DEFLATE entries, longest first; [0, n_inflate_big) are the large ones
	uint32_t n_inflate_big;
	uint32_t n_inflate_huge;   // [0, n_inflate_huge): entries whose serial decode time sets the critical path of a batch
	uint32_t huge_split[2];    // [0, huge_split[0]): the huge entries of at least half the largest one's compressed size, [.., huge_split[1]): a quarter
	                           // (their own groups when the huge streams are few)
	I2SegCtl seg;              // segmented decode of the huge entries (device arrays; null when there are none)
	uint64_t sym_elems;        // symbol buffer the parallel execution of the huge streams may need
	uint64_t *d_tok_ofs;       // two-phase inflate: scratch offset of every list slot (+ end), bytes
	uint64_t tok_bytes;
	I2TokRes *d_tokres;
	uint32_t *d_fb_list;       // entries phase A hands to k_inflate
	uint32_t *d_zstd_list, n_zstd;
	OtzCrcChunk *d_zchunks;    // CRC chunks of the method-93 entries (reference containers and real Zstandard frames)
	uint32_t n_zchunks;
	uint32_t *d_d64_list, n_d64;   // Deflate64 entries (method 9), longest first; [0, n_d64_big) are the large ones
	uint32_t n_d64_big;
	uint32_t *d_xz_list, n_xz;     // XZ entries (method 95), longest first
	XzEnt *d_xz_ent;               // per list slot: its range of the segment table, the walk's and the segments' verdicts
	XzSeg *d_xz_segs;              // segment table: floor(uncomp_size / XZ_SEG_MIN) + 1 slots per entry, in list order
	uint32_t n_xz_slots;
	uint64_t *d_ztok_ofs;      // two-phase Zstandard: token scratch offset of every method-93 list slot (+ end)
	uint64_t ztok_bytes;
	I2TokRes *d_ztokres;
	uint32_t *d_counter;
	uint64_t out_bytes_needed;
};

// ---------------------------------------------------------------- CRC tables (host)
static uint32_t h_mulmod(uint32_t a, uint32_t b) {
	uint32_t p = 0;
	for (int i = 0; i < 32; i++) {
		if (a & (0x80000000u >> i)) {
			p ^= b;
		}
		b = (b >> 1) ^ ((b & 1u) ? OTZ_CRC_POLY : 0u);
	}
	return p;
}

static void build_crc_tables(OtzCrcTables *t) {
	for (uint32_t i = 0; i < 256; i++) {
		uint32_t c = i;
		for (int k = 0; k < 8; k++) {
			c = (c & 1) ? OTZ_CRC_POLY ^ (c >> 1) : c >> 1;
		}
		t->t0[i] = c;
	}
	// z[k][b] = state contribution of byte b followed by k zero bytes
	std::vector<uint32_t> cur(t->t0, t->t0 + 256);
	for (int k = 0; k <= 511; k++) {
		if (k >= 496) {
			memcpy(t->skip[511 - k], cur.data(), 1024);  // skip[i] = z[511 - i]
		}
		for (int b = 0; b < 256; b++) {
			cur[b] = (cur[b] >> 8) ^ t->t0[cur[b] & 0xFF];
		}
	}
	t->x2n[0] = 0x40000000u;  // x^1
	for (int k = 1; k < 32; k++) {
		t->x2n[k] = h_mulmod(t->x2n[k - 1], t->x2n[k - 1]);
	}
	// x^8 and its inverse x^(2^32-1-8)
	uint32_t x8 = t->x2n[3], x8inv = 0x80000000u;
	{
		uint64_t ex = 0xFFFFFFFFull - 8ull;
		for (int k = 0; ex; k++, ex >>= 1) {
			if (ex & 1) {
				x8inv = h_mulmod(x8inv, t->x2n[k & 31]);
			}
		}
	}
	const int nxp = (int)(sizeof(t->xp8) / sizeof(t->xp8[0]));
	t->xp8[OTZ_XP8_BIAS] = 0x80000000u;
	for (int k = OTZ_XP8_BIAS + 1; k < nxp; k++) {
		t->xp8[k] = h_mulmod(t->xp8[k - 1], x8);
	}
	for (int k = OTZ_XP8_BIAS - 1; k >= 0; k--) {
		t->xp8[k] = h_mulmod(t->xp8[k + 1], x8inv);
	}
	t->x_inv_fold = 0x80000000u;
	for (int k = 0; k < 512 * FOLD_K; k++) {
		t->x_inv_fold = h_mulmod(t->x_inv_fold, x8inv);
	}
}

// ---------------------------------------------------------------- context
extern "C" const char *otz_last_error(void) { return g_err; }

// debug build (-DOTZ_BOUNDS_CHECK, `make debug`): violations counted by the OTZ_CHK sites of the kernels since the library was
// loaded; returns the number of counters, -1 in the release build (no checks compiled in)
extern "C" int otz_debug_violations(uint64_t *out, int cap) {
#ifdef OTZ_BOUNDS_CHECK
	unsigned long long h[OTZ_CHK_SLOTS];
	if (cudaMemcpyFromSymbol(h, g_otz_violations, sizeof(h)) != cudaSuccess) {
		return fail_cuda(cudaGetLastError(), "cudaMemcpyFromSymbol(g_otz_violations)");
	}
	for (int i = 0; i < OTZ_CHK_SLOTS && i < cap; i++) {
		out[i] = h[i];
	}
	return OTZ_CHK_SLOTS;
#else
	(void)out;
	(void)cap;
	return -1;
#endif
}

extern "C" int otz_device_count(void) {
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) {
		cudaGetLastError();
		return 0;
	}
	return n;
}

extern "C" int otz_ctx_create(int device, otz_ctx **out) {
	if (!out) {
		return OTZ_ERR_ARG;
	}
	*out = nullptr;
	CK(cudaSetDevice(device));
	otz_ctx *c = new (std::nothrow) otz_ctx();
	if (!c) {
		return OTZ_ERR_NOMEM;
	}
	c->device = device;   // (value-initialised by new otz_ctx(): every field is zero)
	cudaDeviceProp prop;
	CK(cudaGetDeviceProperties(&prop, device));
	c->sm_count = prop.multiProcessorCount;
	CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
	CK(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
	CK(cudaStreamCreateWithFlags(&c->stream3, cudaStreamNonBlocking));
	CK(cudaStreamCreateWithFlags(&c->stream4, cudaStreamNonBlocking));
	CK(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
	CK(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
	CK(cudaEventCreateWithFlags(&c->ev_join3, cudaEventDisableTiming));
	CK(cudaEventCreateWithFlags(&c->ev_join4, cudaEventDisableTiming));
	for (int k = 0; k < 2; k++) {
		CK(cudaStreamCreateWithFlags(&c->stream_d64[k], cudaStreamNonBlocking));
		CK(cudaEventCreateWithFlags(&c->ev_d64_join[k], cudaEventDisableTiming));
	}
	CK(cudaEventCreateWithFlags(&c->ev_d64_fork, cudaEventDisableTiming));
	CK(cudaStreamCreateWithFlags(&c->stream_xz, cudaStreamNonBlocking));
	CK(cudaEventCreateWithFlags(&c->ev_xz_fork, cudaEventDisableTiming));
	CK(cudaEventCreateWithFlags(&c->ev_xz_join, cudaEventDisableTiming));
	CK(cudaEventCreate(&c->ev0));
	CK(cudaEventCreate(&c->ev1));
	for (auto &slot : c->pev) {
		for (auto &e : slot) {
			CK(cudaEventCreate(&e));
		}
	}
	{
		ZseTables zt;   // Zstandard encoder tables (predefined distributions) -> constant memory of this device
		zse_build_tables(&zt);
		CK(cudaMemcpyToSymbol(c_zse, &zt, sizeof(zt)));
	}
	OtzCrcTables *h = new OtzCrcTables();
	build_crc_tables(h);
	CK(cudaMalloc(&c->d_tabs, sizeof(OtzCrcTables)));
	CK(cudaMemcpy(c->d_tabs, h, sizeof(OtzCrcTables), cudaMemcpyHostToDevice));
	delete h;
	const char *t = getenv("OTZ_INFLATE_TILE");   // 0 / unset: chosen per batch
	c->inflate_tile = t ? atoi(t) : 0;
	t = getenv("OTZ_INFLATE_RING");
	c->inflate_ring = t ? atoi(t) : 0;
	t = getenv("OTZ_INFLATE_MODE");
	c->inflate_mode = (t && !strcmp(t, "legacy")) ? 1 : 0;
	t = getenv("OTZ_HUGE_MODE");
	c->huge_legacy = (t && !strcmp(t, "legacy")) ? 1 : 0;
	t = getenv("OTZ_SEG_EXEC");
	c->seg_serial = (t && !strcmp(t, "serial")) ? 1 : 0;
	t = getenv("OTZ_SEG_PAR_RING");
	c->seg_ring = t ? atoi(t) : 4096;
	t = getenv("OTZ_SEG_SYM_LIMIT");
	c->sym_limit = t ? strtoull(t, nullptr, 0) : ~0ull;
	t = getenv("OTZ_LZ_RING");
	c->lz_ring = t ? atoi(t) : 4096;
	*out = c;
	return OTZ_SUCCESS;
}

static void aes_destroy(otz_ctx *c);
extern "C" void otz_ctx_destroy(otz_ctx *c) {
	if (!c) {
		return;
	}
	cudaSetDevice(c->device);
	cudaStreamSynchronize(c->stream);
	cudaFree(c->d_tabs);
	cudaFree(c->d_flush);
	cudaFree(c->d_arch_cache);
	cudaFree(c->d_out_cache);
	cudaFree(c->d_tok_cache);
	cudaFree(c->d_sym_cache);
	cudaFree(c->d_ztok_cache);
	cudaFree(c->d_spec_tmp);
	aes_destroy(c);
	for (size_t k = 0; k < c->pc_plans.size(); k++) {
		otz_plan_destroy(c->pipe[k & 1], c->pc_plans[k]);
	}
	cudaFreeHost(c->h_res);
	for (auto &pc : c->pipe) {
		otz_ctx_destroy(pc);
	}
	cudaSetDevice(c->device);
	cudaEventDestroy(c->ev0);
	cudaEventDestroy(c->ev1);
	for (auto &slot : c->pev) {
		for (auto &e : slot) {
			cudaEventDestroy(e);
		}
	}
	cudaEventDestroy(c->ev_fork);
	cudaEventDestroy(c->ev_join);
	cudaEventDestroy(c->ev_join3);
	cudaEventDestroy(c->ev_join4);
	cudaEventDestroy(c->ev_d64_fork);
	cudaEventDestroy(c->ev_xz_fork);
	cudaEventDestroy(c->ev_xz_join);
	cudaStreamDestroy(c->stream_xz);
	for (int k = 0; k < 2; k++) {
		cudaEventDestroy(c->ev_d64_join[k]);
		cudaStreamDestroy(c->stream_d64[k]);
	}
	cudaStreamDestroy(c->stream4);
	cudaStreamDestroy(c->stream3);
	cudaStreamDestroy(c->stream2);
	cudaStreamDestroy(c->stream);
	delete c;
}

extern "C" int otz_sm_count(otz_ctx *c) { return c ? c->sm_count : 0; }
extern "C" int otz_pci_bus_id(otz_ctx *c, char *buf, int len) {
	CK(cudaDeviceGetPCIBusId(buf, len, c->device));
	return OTZ_SUCCESS;
}
extern "C" uint64_t otz_launch_count(otz_ctx *c) { return c ? c->launches : 0; }

// ---------------------------------------------------------------- memory
extern "C" int otz_dev_alloc(otz_ctx *c, uint64_t bytes, void **dptr) {
	if (!c || !dptr) {
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	CK(cudaMalloc(dptr, bytes + 64));
	return OTZ_SUCCESS;
}
extern "C" int otz_dev_free(otz_ctx *c, void *dptr) {
	if (!c) {
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	CK(cudaFree(dptr));
	return OTZ_SUCCESS;
}
extern "C" int otz_host_alloc(uint64_t bytes, void **hptr) {
	CK(cudaHostAlloc(hptr, bytes ? bytes : 1, cudaHostAllocPortable));   // (pinned for every device: the multi-GPU call shares one arena)
	return OTZ_SUCCESS;
}
extern "C" int otz_host_free(void *hptr) {
	CK(cudaFreeHost(hptr));
	return OTZ_SUCCESS;
}
extern "C" int otz_h2d(otz_ctx *c, void *dptr, const void *hptr, uint64_t bytes) {
	CK(cudaSetDevice(c->device));
	CK(cudaMemcpyAsync(dptr, hptr, bytes, cudaMemcpyHostToDevice, c->stream));
	return OTZ_SUCCESS;
}
extern "C" int otz_d2h(otz_ctx *c, void *hptr, const void *dptr, uint64_t bytes) {
	CK(cudaSetDevice(c->device));
	CK(cudaMemcpyAsync(hptr, dptr, bytes, cudaMemcpyDeviceToHost, c->stream));
	return OTZ_SUCCESS;
}
extern "C" int otz_dev_memset(otz_ctx *c, void *dptr, int value, uint64_t bytes) {
	CK(cudaSetDevice(c->device));
	CK(cudaMemsetAsync(dptr, value, bytes, c->stream));
	return OTZ_SUCCESS;
}
extern "C" int otz_sync(otz_ctx *c) {
	CK(cudaSetDevice(c->device));
	CK(cudaStreamSynchronize(c->stream));
	return OTZ_SUCCESS;
}

// ---------------------------------------------------------------- timing
extern "C" int otz_timer_start(otz_ctx *c) {
	CK(cudaSetDevice(c->device));
	CK(cudaEventRecord(c->ev0, c->stream));
	return OTZ_SUCCESS;
}
extern "C" int otz_timer_stop(otz_ctx *c, float *ms) {
	CK(cudaSetDevice(c->device));
	CK(cudaEventRecord(c->ev1, c->stream));
	CK(cudaEventSynchronize(c->ev1));
	CK(cudaEventElapsedTime(ms, c->ev0, c->ev1));
	return OTZ_SUCCESS;
}
extern "C" int otz_profile_enable(otz_ctx *c, int on) {
	c->profile = on;
	c->prof_runs = 0;
	return OTZ_SUCCESS;
}
extern "C" int otz_profile_runs(otz_ctx *c) { return (int)c->prof_runs; }
extern "C" int otz_profile_get(otz_ctx *c, int run, float *r, float *d, float *k, float *f) {
	CK(cudaSetDevice(c->device));
	if (run < 0 || (uint32_t)run >= c->prof_runs || c->prof_runs - (uint32_t)run > OTZ_PROF_SLOTS) {
		return OTZ_ERR_ARG;
	}
	cudaEvent_t *ev = c->pev[run % OTZ_PROF_SLOTS];
	CK(cudaEventSynchronize(ev[4]));
	float *dst[4] = { r, d, k, f };
	for (int i = 0; i < 4; i++) {
		if (dst[i]) {
			CK(cudaEventElapsedTime(dst[i], ev[i], ev[i + 1]));
		}
	}
	return OTZ_SUCCESS;
}

__global__ void k_flush_fill(uint4 *p, uint64_t n, uint32_t v) {
	for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
		p[i] = make_uint4(v, v, v, v);
	}
}
extern "C" int otz_flush_l2(otz_ctx *c) {
	CK(cudaSetDevice(c->device));
	if (!c->d_flush) {
		c->flush_bytes = 256ull << 20;  // 2x the 126 MB L2
		CK(cudaMalloc(&c->d_flush, c->flush_bytes));
	}
	k_flush_fill<<<c->sm_count * 4, 256, 0, c->stream>>>(reinterpret_cast<uint4 *>(c->d_flush), c->flush_bytes / 16, (uint32_t)c->launches);
	CK(cudaGetLastError());
	return OTZ_SUCCESS;
}

// ---------------------------------------------------------------- read path
static uint32_t crc_ctas_per_sm() {
	static int per_sm = 0;
	if (!per_sm) {
		if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_crc_chunks, 256, 0) != cudaSuccess || per_sm < 1) {
			per_sm = 1;
		}
	}
	return (uint32_t)per_sm;
}

template <typename T>
static int upload(T **d, const std::vector<T> &h, cudaStream_t s) {
	*d = nullptr;
	CK(cudaMalloc(d, std::max<size_t>(h.size(), 1) * sizeof(T)));
	if (!h.empty()) {
		CK(cudaMemcpyAsync(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s));
	}
	return OTZ_SUCCESS;
}

extern "C" void otz_plan_destroy(otz_ctx *c, otz_plan *p) {
	if (!p) {
		return;
	}
	if (c) {
		cudaSetDevice(c->device);
		cudaStreamSynchronize(c->stream);
	}
	cudaFree(p->d_ents);
	cudaFree(p->d_est);
	cudaFree(p->d_status);
	cudaFree(p->d_acc);
	cudaFree(p->d_crc);
	cudaFree(p->d_produced);
	cudaFree(p->d_chunks);
	cudaFree(p->d_inflate_list);
	cudaFree(p->seg.count);
	cudaFree(p->seg.start);
	cudaFree(p->seg.res);
	cudaFree(p->seg.live);
	cudaFree(p->seg.nlive);
	cudaFree(p->seg.seg_status);
	cudaFree(p->seg.par);
	cudaFree(p->seg.par_items);
	cudaFree(p->seg.n_par);
	cudaFree(p->seg.sym_start);
	cudaFree(p->seg.out_start);
	cudaFree(p->d_tok_ofs);
	cudaFree(p->d_tokres);
	cudaFree(p->d_fb_list);
	cudaFree(p->d_zstd_list);
	cudaFree(p->d_zchunks);
	cudaFree(p->d_d64_list);
	cudaFree(p->d_xz_list);
	cudaFree(p->d_xz_ent);
	cudaFree(p->d_xz_segs);
	cudaFree(p->d_ztok_ofs);
	cudaFree(p->d_ztokres);
	cudaFree(p->d_counter);
	delete p;
}

extern "C" int otz_plan_create(otz_ctx *c, const otz_entry *ents, uint32_t n, const otz_extract_opts *opts, otz_plan **out) {
	if (!c || !out || (n && !ents) || !opts) {
		return OTZ_ERR_ARG;
	}
	*out = nullptr;
	CK(cudaSetDevice(c->device));
	otz_plan *p = new (std::nothrow) otz_plan();
	if (!p) {
		return OTZ_ERR_NOMEM;
	}
	memset(p, 0, sizeof(*p));
	p->n = n;
	p->opts = *opts;
	for (uint32_t i = 0; i < n; i++) {
		// a chunk row names its parent row in crc32: the decoders write status[parent] when a chunk fails
		if ((ents[i].flags & OTZ_EF_CHUNK) && (ents[i].crc32 >= n || !(ents[ents[i].crc32].flags & OTZ_EF_PARENT))) {
			delete p;
			snprintf(g_err, sizeof(g_err), "entry table row %u: chunk row without a parent row", i);
			return OTZ_ERR_ARG;
		}
	}
	// Work lists.  CRC chunks: STORE entries first (they are also the copy list), then the rest.
	std::vector<OtzCrcChunk> chunks;
	std::vector<uint32_t> infl, zst, d64, xz;
	uint64_t need = 0;
	for (int pass = 0; pass < 2; pass++) {
		for (uint32_t i = 0; i < n; i++) {
			const bool is_store = ents[i].method == OTZ_M_STORE;
			if ((pass == 0) != is_store || ents[i].method == OTZ_M_ZSTD || (ents[i].flags & OTZ_EF_CHUNK)) {
				continue;   // method 93 has its own chunk list (below); chunk rows are CRC'd through their parent
			}
			const uint32_t nc = (uint32_t)(((uint64_t)ents[i].uncomp_size + OTZ_CRC_CHUNK - 1) / OTZ_CRC_CHUNK);
			for (uint32_t k = 0; k < nc; k++) {
				chunks.push_back(OtzCrcChunk{ i, k });
			}
		}
		if (pass == 0) {
			p->n_store_chunks = (uint32_t)chunks.size();
		}
	}
	for (uint32_t i = 0; i < n; i++) {
		if (ents[i].method == OTZ_M_DEFLATE) {
			if (!(ents[i].flags & OTZ_EF_PARENT)) {
				infl.push_back(i);   // a parent row is decoded through its chunk rows
			}
		} else if (ents[i].method == OTZ_M_ZSTD) {
			zst.push_back(i);
		} else if (ents[i].method == OTZ_M_DEFLATE64 && !(ents[i].flags & OTZ_EF_CHUNK)) {
			d64.push_back(i);   // never on the two-phase path: its 32-bit records hold neither 64 KiB distances nor long lengths
		} else if (ents[i].method == OTZ_M_XZ && !(ents[i].flags & OTZ_EF_CHUNK)) {
			xz.push_back(i);
		}
		if (!(opts->verify_only && ents[i].method == OTZ_M_STORE)) {
			need = std::max<uint64_t>(need, ents[i].out_ofs + ents[i].uncomp_size);
		}
	}
	std::vector<OtzCrcChunk> zchunks;
	for (uint32_t i : zst) {
		const uint32_t nc = (uint32_t)(((uint64_t)ents[i].uncomp_size + OTZ_CRC_CHUNK - 1) / OTZ_CRC_CHUNK);
		for (uint32_t k = 0; k < nc; k++) {
			zchunks.push_back(OtzCrcChunk{ i, k });
		}
	}
	p->n_zchunks = (uint32_t)zchunks.size();
	// longest streams first: the tail of the batch is then made of short ones
	// large entries first (they get the 16 KiB ring kernel), inside each class longest streams first
	const uint32_t big_bytes = 256u * 1024u;
	const char *hb = getenv("OTZ_HUGE_BYTES");
	const uint32_t huge_bytes = hb ? (uint32_t)strtoul(hb, nullptr, 0) : 1024u * 1024u;
	// (the segmented decode keeps bit positions in 32 bits: streams of 512 MiB and more stay on the other paths)
	auto is_huge = [&](uint32_t i) { return ents[i].uncomp_size >= huge_bytes && ents[i].comp_size < (1u << 29); };
	auto cls = [&](uint32_t i) { return is_huge(i) ? 2 : ents[i].uncomp_size >= big_bytes ? 1 : 0; };
	std::stable_sort(infl.begin(), infl.end(), [&](uint32_t a, uint32_t b) {
		const int ca = cls(a), cb = cls(b);
		return ca != cb ? ca > cb : ents[a].comp_size > ents[b].comp_size;
	});
	p->n_inflate_big = 0;
	p->n_inflate_huge = 0;
	for (uint32_t i : infl) {
		p->n_inflate_big += ents[i].uncomp_size >= big_bytes;
		p->n_inflate_huge += is_huge(i);
	}
	// Deflate64: sized as the one-kernel DEFLATE dispatch sizes its launches (large entries first, longest first)
	std::stable_sort(d64.begin(), d64.end(), [&](uint32_t a, uint32_t b) {
		const bool ba = ents[a].uncomp_size >= big_bytes, bb = ents[b].uncomp_size >= big_bytes;
		return ba != bb ? ba : ents[a].comp_size > ents[b].comp_size;
	});
	p->n_d64_big = 0;
	for (uint32_t i : d64) {
		p->n_d64_big += ents[i].uncomp_size >= big_bytes;
	}
	p->n_d64 = (uint32_t)d64.size();
	// XZ: longest first; every entry gets the segment slots its declared size can need
	std::stable_sort(xz.begin(), xz.end(), [&](uint32_t a, uint32_t b) { return ents[a].comp_size > ents[b].comp_size; });
	std::vector<XzEnt> xe(xz.size());
	uint64_t xz_slots = 0;
	for (size_t k = 0; k < xz.size(); k++) {
		xe[k].first = (uint32_t)xz_slots;
		xe[k].cap = ents[xz[k]].uncomp_size / XZ_SEG_MIN + 1u;
		xz_slots += xe[k].cap;
	}
	p->n_xz = (uint32_t)xz.size();
	p->n_xz_slots = (uint32_t)xz_slots;
	p->n_chunks = (uint32_t)chunks.size();
	p->n_inflate = (uint32_t)infl.size();
	p->n_zstd = (uint32_t)zst.size();
	p->out_bytes_needed = need;
	int rc;
	std::vector<otz_entry> ev(ents, ents + n);
	// two-phase inflate: worst-case token scratch per list slot
	std::vector<uint64_t> tofs(infl.size() + 1);
	tofs[0] = 0;
	for (size_t k = 0; k < infl.size(); k++) {
		tofs[k + 1] = tofs[k] + i2_scratch_bytes(ents[infl[k]].uncomp_size);
	}
	p->tok_bytes = tofs.back();
	if (p->n_inflate && ((rc = upload(&p->d_tok_ofs, tofs, c->stream)) ||
			cudaMalloc(&p->d_tokres, infl.size() * sizeof(I2TokRes)) != cudaSuccess ||
			cudaMalloc(&p->d_fb_list, infl.size() * 4) != cudaSuccess)) {
		otz_plan_destroy(c, p);
		return rc ? rc : fail_cuda(cudaGetLastError(), "cudaMalloc(two-phase inflate lists)");
	}
	if (p->n_inflate_huge && p->n_inflate_huge <= 4096u) {
		const size_t nh = p->n_inflate_huge, ns = nh * I2_MAXSEG;
		// size groups of the few-streams regime (dispatch_inflate3), in percent of the largest stream's compressed size (75 / 50
		// and 85 / 60 measured the same on a 1,250-entry shard: the chains are bound by the latency of the largest stream)
		const uint64_t split_pct[2] = { 50u, 25u };
		for (size_t h = 0; h < nh; h++) {
			p->huge_split[0] += (uint64_t)ents[infl[h]].comp_size * 100u >= (uint64_t)ents[infl[0]].comp_size * split_pct[0];   // (the list is sorted by compressed size)
			p->huge_split[1] += (uint64_t)ents[infl[h]].comp_size * 100u >= (uint64_t)ents[infl[0]].comp_size * split_pct[1];
			// symbols of the stream + markers in front of every segment (a stream with more segments than estimated here is
			// executed by one warp)
			p->sym_elems += (uint64_t)ents[infl[h]].uncomp_size +
				(uint64_t)(I2_PREWIN + 16u) * std::min<uint64_t>(I2_MAXSEG, 2u + ents[infl[h]].uncomp_size / I3_SEG_MIN);
		}
		if (cudaMalloc(&p->seg.count, nh * 4) != cudaSuccess || cudaMalloc(&p->seg.start, ns * 4) != cudaSuccess ||
			cudaMalloc(&p->seg.res, ns * sizeof(I2SegRes)) != cudaSuccess || cudaMalloc(&p->seg.live, ns * 4) != cudaSuccess ||
			cudaMalloc(&p->seg.nlive, nh * 4) != cudaSuccess || cudaMalloc(&p->seg.seg_status, nh * 4) != cudaSuccess ||
			cudaMalloc(&p->seg.par, nh * 4) != cudaSuccess || cudaMalloc(&p->seg.par_items, ns * 4) != cudaSuccess ||
			cudaMalloc(&p->seg.n_par, 16) != cudaSuccess || cudaMalloc(&p->seg.sym_start, ns * 8) != cudaSuccess ||
			cudaMalloc(&p->seg.out_start, ns * 4) != cudaSuccess) {
			otz_plan_destroy(c, p);
			return fail_cuda(cudaGetLastError(), "cudaMalloc(segment tables)");
		}
	}
	if ((rc = upload(&p->d_ents, ev, c->stream)) || (rc = upload(&p->d_chunks, chunks, c->stream)) ||
		(rc = upload(&p->d_inflate_list, infl, c->stream)) || (rc = upload(&p->d_zstd_list, zst, c->stream)) ||
		(rc = upload(&p->d_zchunks, zchunks, c->stream)) || (rc = upload(&p->d_d64_list, d64, c->stream)) ||
		(rc = upload(&p->d_xz_list, xz, c->stream)) || (rc = upload(&p->d_xz_ent, xe, c->stream))) {
		otz_plan_destroy(c, p);
		return rc;
	}
	const size_t n1 = std::max<uint32_t>(n, 1);
	if (cudaMalloc(&p->d_est, n1 * sizeof(OtzEntryState)) != cudaSuccess || cudaMalloc(&p->d_status, n1 * 4) != cudaSuccess ||
		cudaMalloc(&p->d_acc, n1 * 4) != cudaSuccess || cudaMalloc(&p->d_crc, n1 * 4) != cudaSuccess ||
		cudaMalloc(&p->d_produced, n1 * 4) != cudaSuccess ||
		cudaMalloc(&p->d_xz_segs, std::max<uint64_t>(xz_slots, 1) * sizeof(XzSeg)) != cudaSuccess ||
		cudaMalloc(&p->d_counter, 256) != cudaSuccess) {
		otz_plan_destroy(c, p);
		return fail_cuda(cudaGetLastError(), "cudaMalloc(plan)");
	}
	if (p->n_zstd) {
		std::vector<uint64_t> zofs(zst.size() + 1);
		zofs[0] = 0;
		for (size_t k = 0; k < zst.size(); k++) {
			zofs[k + 1] = zofs[k] + zs_scratch_bytes(ents[zst[k]].uncomp_size);
		}
		p->ztok_bytes = zofs.back();
		if ((rc = upload(&p->d_ztok_ofs, zofs, c->stream)) || cudaMalloc(&p->d_ztokres, zst.size() * (sizeof(I2TokRes) + 8)) != cudaSuccess   /* + the verdicts of the two tokenizers */) {
			otz_plan_destroy(c, p);
			return rc ? rc : fail_cuda(cudaGetLastError(), "cudaMalloc(two-phase zstd lists)");
		}
		CK(cudaStreamSynchronize(c->stream));   // zofs dies here
	}
	CK(cudaMemsetAsync(p->d_counter, 0, 256, c->stream));
	CK(cudaStreamSynchronize(c->stream));  // the host vectors die here
	*out = p;
	return OTZ_SUCCESS;
}

template <int G, int W, bool D64 = false>
static int launch_inflate(otz_ctx *c, otz_plan *p, const uint8_t *d_archive, uint8_t *d_out, const uint32_t *d_list, uint32_t count,
	uint32_t *d_work, cudaStream_t st, const uint32_t *d_count) {
	const int threads = 8 * G;   // 8 streams per CTA
	const size_t smem = 8 * sizeof(InflateSmemV2<G, W>);
	static bool attr_done = false;
	if (!attr_done) {
		CK(cudaFuncSetAttribute(k_inflate<G, W, D64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		attr_done = true;
	}
	int per_sm = 0;
	CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_inflate<G, W, D64>, threads, smem));
	if (per_sm < 1) {
		snprintf(g_err, sizeof(g_err), "k_inflate<%d,%d> does not fit an SM (%zu bytes of shared memory)", G, W, smem);
		return OTZ_ERR_CUDA;
	}
	const uint32_t tiles_per_cta = threads / G;
	uint32_t grid = (uint32_t)(c->sm_count * per_sm);
	const uint32_t want = (count + tiles_per_cta - 1) / tiles_per_cta;
	grid = std::max(1u, std::min(grid, want));
	k_inflate<G, W, D64><<<grid, threads, smem, st>>>(d_archive, d_out, p->d_ents, p->d_est, p->d_status, d_list, count, d_work, p->d_produced, d_count);
	c->launches++;
	CK(cudaGetLastError());
	return OTZ_SUCCESS;
}

template <bool D64 = false>
static int launch_inflate_cfg(otz_ctx *c, otz_plan *p, const uint8_t *d_archive, uint8_t *d_out, int g, int w, uint32_t first, uint32_t count,
	int slot /* word of d_counter used as the work counter */, cudaStream_t st, const uint32_t *d_list = nullptr,
	const uint32_t *d_count = nullptr) {
	if (!d_list) {
		d_list = (D64 ? p->d_d64_list : p->d_inflate_list) + first;
	}
#define OTZ_INF_CASE(G_, W_)        \
	if (g == G_ && w == W_) {       \
		return launch_inflate<G_, W_, D64>(c, p, d_archive, d_out, d_list, count, p->d_counter + slot, st, d_count); \
	}
	OTZ_INF_CASE(32, 16384)
	OTZ_INF_CASE(32, 4096)
	OTZ_INF_CASE(32, 2048)
	OTZ_INF_CASE(16, 4096)
	OTZ_INF_CASE(16, 2048)
	OTZ_INF_CASE(8, 4096)
	OTZ_INF_CASE(8, 2048)
	OTZ_INF_CASE(8, 1024)
	OTZ_INF_CASE(4, 2048)
	OTZ_INF_CASE(4, 1024)
#undef OTZ_INF_CASE
	snprintf(g_err, sizeof(g_err), "unsupported OTZ_INFLATE_TILE/OTZ_INFLATE_RING combination %d/%d", g, w);
	return OTZ_ERR_ARG;
}

// One warp per stream.  The ring size trades per-stream speed (a 16 KiB ring serves ~85% of the back-references
// of text from shared memory, a 2 KiB ring ~35%) against resident streams per SM (10 vs 24).  Large entries set
// the critical path of a batch, so they always get the big ring, on a second stream so that both kernels can
// share the machine; small entries get the big ring only when there are too few of them to fill the SMs.
template <int W>
static int launch_lz(otz_ctx *c, otz_plan *p, uint8_t *d_out, uint32_t first, uint32_t count, cudaStream_t st) {
	auto kern = k_inflate_lz<W, false, false>;
	const int warps = 4;
	const size_t smem = warps * sizeof(I2LzSmem<W>);
	static bool attr_done = false;
	if (!attr_done) {
		CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		attr_done = true;
	}
	int per_sm = 0;
	CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * warps, smem));
	if (per_sm < 1) {
		snprintf(g_err, sizeof(g_err), "k_inflate_lz<%d> does not fit an SM", W);
		return OTZ_ERR_CUDA;
	}
	const uint32_t grid = std::max(1u, std::min((uint32_t)(c->sm_count * per_sm), (count + warps - 1) / warps));
	kern<<<grid, 32 * warps, smem, st>>>(d_out, p->d_ents, p->d_inflate_list + first, count, p->d_counter + 48, c->d_tok_cache,
		p->d_tok_ofs + first, p->d_tokres + first, p->d_status, p->d_produced, I2SegCtl{}, 0u);
	c->launches++;
	CK(cudaGetLastError());
	return OTZ_SUCCESS;
}

// Parallel execution of the chains k_seg_stitch placed in the symbol buffer: one warp per segment over 16-bit symbols,
// then the windows between the segments (one CTA per stream), then symbols -> bytes for everything else.
template <int W>
static int launch_seg_par(otz_ctx *c, otz_plan *p, uint8_t *d_out, const I2SegCtl &sg, cudaStream_t st, uint32_t h0, uint32_t h1, uint32_t *cnt_par,
	uint32_t *cnt_tr) {
	auto kern = k_inflate_lz<W, false, true, true>;
	const int warps = 4;
	const size_t smem = warps * sizeof(I2LzSmem<W, uint16_t>);
	static bool attr_done = false;
	if (!attr_done) {
		CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		attr_done = true;
	}
	int per_sm = 0;
	CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * warps, smem));
	if (per_sm < 1) {
		snprintf(g_err, sizeof(g_err), "k_inflate_lz<%d, symbols> does not fit an SM", W);
		return OTZ_ERR_CUDA;
	}
	kern<<<(uint32_t)(c->sm_count * per_sm), 32 * warps, smem, st>>>(reinterpret_cast<uint8_t *>(c->d_sym_cache), p->d_ents, p->d_inflate_list, 0u, cnt_par,
		c->d_tok_cache, p->d_tok_ofs, p->d_tokres, p->d_status, p->d_produced, sg, 0u);
	k_seg_window<<<h1 - h0, 1024, 0, st>>>(d_out, p->d_ents, p->d_inflate_list, h1, c->d_sym_cache, p->d_status, p->d_produced, sg, h0);
	k_seg_translate<<<(uint32_t)c->sm_count * 4u, I2_TR_THREADS, 0, st>>>(d_out, p->d_ents, p->d_inflate_list, c->d_sym_cache, cnt_tr, sg);
	c->launches += 3;
	CK(cudaGetLastError());
	return OTZ_SUCCESS;
}

// Two-phase inflate, warp-per-stream speculative tokenizer (k_inflate3.cuh): ONE tokenizer launch for every DEFLATE
// stream of the batch (longest first); huge streams come out as segment tables, which k_seg_stitch places in the symbol
// buffer for the parallel execution (second stream), everything else goes to k_inflate_lz; then k_inflate over whatever
// phase A declined (d_counter + 52 counts those entries).
// temp token slots of k_inflate_spec (I3_TMP_BYTES per resident lane; at most 1,024 lanes of these kernels fit an SM): four
// regions, because the tokenizer of the regular streams and those of up to three size groups of huge streams run at once.
// Allocated once per context.
static int reserve_spec_tmp(otz_ctx *c) {
	if (c->d_spec_tmp) {
		return OTZ_SUCCESS;
	}
	c->spec_tmp_region = (uint64_t)c->sm_count * 1024u * I3_TMP_BYTES;
	if (cudaMalloc(&c->d_spec_tmp, 4 * c->spec_tmp_region) != cudaSuccess) {
		c->d_spec_tmp = nullptr;
		return fail_cuda(cudaGetLastError(), "cudaMalloc(tokenizer temp slots)");
	}
	return OTZ_SUCCESS;
}

static int dispatch_inflate3(otz_ctx *c, otz_plan *p, const uint8_t *d_archive, uint8_t *d_out) {
	cudaStream_t s = c->stream, s2 = c->stream2;
	{
		const int rc_ = reserve_spec_tmp(c);
		if (rc_) {
			return rc_;
		}
	}
	static bool attr_done = false;
	const size_t smem1 = I3_WARPS * sizeof(I3Smem<1>), smem4 = sizeof(I3Smem<4>), smem8 = sizeof(I3Smem<8, 16>);
	if (!attr_done) {
		CK(cudaFuncSetAttribute(k_inflate_spec<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
		CK(cudaFuncSetAttribute(k_inflate_spec<1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
		CK(cudaFuncSetAttribute(k_inflate_spec<4, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4));
		CK(cudaFuncSetAttribute(k_inflate_spec<4, 8>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
		CK(cudaFuncSetAttribute(k_inflate_spec<8, 4, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem8));
		CK(cudaFuncSetAttribute(k_inflate_spec<8, 4, 16>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
		CK(cudaFuncSetAttribute(k_inflate_lz<OTZ_SEG_RING, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(4 * sizeof(I2LzSmem<OTZ_SEG_RING>))));
		attr_done = true;
	}
	const uint32_t nh = (p->n_inflate_huge && p->seg.count && !c->huge_legacy) ? p->n_inflate_huge : 0u;
	const uint32_t count = p->n_inflate - nh;
	const char *gs = getenv("OTZ_SPEC_GRID");   // (tests: few groups, so that every group decodes many streams)
	const char *sm_ = getenv("OTZ_SEG_MIN");       // least output bytes of a segment (>= I3_SEG_MIN: the symbol buffer is sized for that)
	const uint32_t seg_min = sm_ ? std::max<uint32_t>(I3_SEG_MIN, (uint32_t)strtoul(sm_, nullptr, 0)) : I3_SEG_MIN;
	bool forked = false;
	// 4-warp CTAs at 64 registers: 8 CTAs = 32 warps per SM (4 CTAs at 104 registers measured 4 % slower on configs[2]).
	// Few huge streams — every one of them a critical path, SMs to spare (a shard of a multi-GPU run, a small archive):
	// 8-warp CTAs, 256 pieces per round, half the rounds per stream (measured: 1,250 entries 21.3 -> 17.4 ms, 5,000 entries
	// 46.7 -> 43.5 ms, 10,000 entries no gain; 4 warps with 1,024-bit pieces: 19.6 ms).  A DEFLATE block of zlib is ~27 KB, about
	// one such round: more lanes would idle.
	const bool wide = nh && ((nh <= (uint32_t)c->sm_count * 16u && !getenv("OTZ_SPEC_NO_WIDE")) || getenv("OTZ_SPEC_FORCE_WIDE"));
	// In that regime the huge streams are also cut into up to THREE groups by size, each with its own chain tokenizer -> stitch ->
	// segment execution -> window -> translate on its own CUDA stream: group 0 = the streams of at least half the largest
	// one's compressed size (their tokenizer runs ~10 ms for a 16 MiB entry whatever else happens), group 1 = down to a
	// quarter, group 2 = the rest, whose segments are already executing while the larger ones are still being tokenized
	// (1,250 entries: 17.6 -> 14.4 ms with two groups).
	struct Grp {
		uint32_t h0, h1;
		cudaStream_t st;
		cudaEvent_t join;
		uint32_t c_spec, c_seglz, c_par, c_tr;   // words of d_counter
		uint32_t par_slot;
	} grp[3] = { { 0u, nh, s2, c->ev_join, 57u, 58u, 60u, 61u, 0u }, { 0u, 0u, c->stream3, c->ev_join3, 40u, 41u, 42u, 43u, 1u },
		{ 0u, 0u, c->stream4, c->ev_join4, 44u, 45u, 46u, 47u, 2u } };
	uint32_t n_grp = nh ? 1u : 0u;
	// (also with many huge streams, as far as the plan knows the cuts: while the segments of one group are executed — bound by
	// instruction issue — the window chain (latency) and the translation (DRAM) of another run next to them: configs[2] as
	// named 241 -> 246 GB/s)
	if (nh && (wide || nh <= 4096u) && !getenv("OTZ_SPEC_ONE_GROUP")) {
		const char *mg = getenv("OTZ_SPEC_GROUPS");
		const uint32_t max_grp = mg ? (uint32_t)atoi(mg) : 3u;
		uint32_t cut[2] = { p->huge_split[0], p->huge_split[1] };
		uint32_t lo = 0;
		n_grp = 0;
		for (uint32_t g = 0; g < 2 && n_grp + 1 < max_grp; g++) {
			if (cut[g] > lo && cut[g] < nh) {
				grp[n_grp].h0 = lo;
				grp[n_grp].h1 = cut[g];
				lo = cut[g];
				n_grp++;
			}
		}
		grp[n_grp].h0 = lo;
		grp[n_grp].h1 = nh;
		n_grp++;
	}
	// OTZ_INFLATE_TRACE=1: a timeline of the chains of one run, printed to stderr (a diagnostic: it waits for the run)
	const bool itrace = getenv("OTZ_INFLATE_TRACE") != nullptr;
	cudaEvent_t tev[12] = {};
	if (itrace) {
		for (int i = 0; i < 12; i++) {
			CK(cudaEventCreate(&tev[i]));
		}
		CK(cudaEventRecord(tev[0], s));
	}
	I2SegCtl sg = p->seg;
	if (nh) {
		// huge streams: the warps of a CTA decode one stream together; second (and third) stream, next to the warp-per-stream kernel
		sg.sym_top = reinterpret_cast<unsigned long long *>(p->d_counter + 62);
		sg.out_mis = (uint32_t)(reinterpret_cast<uint64_t>(d_out) & 15u);
		sg.sym_cap = 0;
		if (!c->seg_serial && p->sym_elems) {
			if (p->sym_elems > c->sym_cache_elems) {
				CK(cudaStreamSynchronize(c->stream));
				CK(cudaStreamSynchronize(s2));
				CK(cudaStreamSynchronize(c->stream3));
				CK(cudaStreamSynchronize(c->stream4));
				cudaFree(c->d_sym_cache);
				c->d_sym_cache = nullptr;
				c->sym_cache_elems = 0;
				if (cudaMalloc(&c->d_sym_cache, p->sym_elems * 2 + 64) == cudaSuccess) {
					c->sym_cache_elems = p->sym_elems;
				} else {
					cudaGetLastError();
				}
			}
			sg.sym_cap = c->d_sym_cache ? std::min<uint64_t>(p->sym_elems, c->sym_limit) : 0;
		}
		CK(cudaEventRecord(c->ev_fork, s));
		auto kern4 = wide ? k_inflate_spec<8, 4, 16> : k_inflate_spec<4, 8>;
		const size_t smem4x = wide ? smem8 : smem4;
		const int thr4 = wide ? 256 : 128;
		int per_sm4 = 0;
		CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm4, kern4, thr4, smem4x));
		if (per_sm4 < 1) {
			snprintf(g_err, sizeof(g_err), "k_inflate_spec for huge streams does not fit an SM (%zu bytes of shared memory)", smem4x);
			return OTZ_ERR_CUDA;
		}
		for (uint32_t g = 0; g < n_grp; g++) {
			const Grp &G = grp[g];
			CK(cudaStreamWaitEvent(G.st, c->ev_fork, 0));
			const uint32_t ng = G.h1 - G.h0;
			const uint32_t grid4 = gs ? (uint32_t)atoi(gs) : std::max(1u, std::min((uint32_t)(c->sm_count * per_sm4), ng));
			kern4<<<grid4, thr4, smem4x, G.st>>>(d_archive, p->d_ents, p->d_est, p->d_status, p->d_inflate_list, G.h0, G.h1, p->d_counter + G.c_spec,
				c->d_tok_cache, p->d_tok_ofs, p->d_tokres, p->d_fb_list, p->d_counter + 52, nh, p->seg, seg_min, c->d_spec_tmp + (1u + g) * c->spec_tmp_region);
			c->launches++;
			CK(cudaGetLastError());
			if (itrace) {
				CK(cudaEventRecord(tev[1 + g], G.st));
			}
		}
	}
	// few streams: a warp per stream leaves the machine idle while every stream waits for its own serial rounds — then the
	// regular streams get a 4-warp CTA each as well (128 pieces per round; configs[0] as written: 1,000 streams on 148 SMs)
	if (count && count <= (uint32_t)c->sm_count * 8u && !getenv("OTZ_SPEC_NO_WIDE")) {
		int per_sm4 = 0;
		auto kern4 = k_inflate_spec<4, 8>;
		CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm4, kern4, 128, smem4));
		const uint32_t grid4 = gs ? (uint32_t)atoi(gs) : std::max(1u, std::min((uint32_t)(c->sm_count * std::max(per_sm4, 1)), count));
		kern4<<<grid4, 128, smem4, s>>>(d_archive, p->d_ents, p->d_est, p->d_status, p->d_inflate_list, nh, p->n_inflate, p->d_counter,
			c->d_tok_cache, p->d_tok_ofs, p->d_tokres, p->d_fb_list, p->d_counter + 52, nh, p->seg, seg_min, c->d_spec_tmp);
		c->launches++;
		CK(cudaGetLastError());
	} else if (count) {
		int per_sm = 0;
		CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_inflate_spec<1>, 32 * I3_WARPS, smem1));
		if (per_sm < 1) {
			snprintf(g_err, sizeof(g_err), "k_inflate_spec<1> does not fit an SM (%zu bytes of shared memory)", smem1);
			return OTZ_ERR_CUDA;
		}
		const uint32_t grid = gs ? (uint32_t)atoi(gs) : std::max(1u, std::min((uint32_t)(c->sm_count * per_sm), (count + I3_WARPS - 1) / I3_WARPS));
		k_inflate_spec<1><<<grid, 32 * I3_WARPS, smem1, s>>>(d_archive, p->d_ents, p->d_est, p->d_status, p->d_inflate_list, nh, p->n_inflate, p->d_counter,
			c->d_tok_cache, p->d_tok_ofs, p->d_tokres, p->d_fb_list, p->d_counter + 52, nh, p->seg, seg_min, c->d_spec_tmp);
		c->launches++;
		CK(cudaGetLastError());
	}
	for (uint32_t g = 0; g < n_grp; g++) {
		const Grp &G = grp[g];
		const uint32_t ng = G.h1 - G.h0;
		I2SegCtl sgg = sg;
		sgg.n_par = p->seg.n_par + G.par_slot;
		sgg.par_items = p->seg.par_items + (size_t)G.h0 * I2_MAXSEG;
		CK(cudaMemsetAsync(sgg.n_par, 0, 4, G.st));
		CK(cudaMemsetAsync(p->seg.nlive + G.h0, 0, ng * 4, G.st));
		CK(cudaMemsetAsync(p->seg.par + G.h0, 0, ng * 4, G.st));
		k_seg_stitch<<<(ng + 63) / 64, 64, 0, G.st>>>(p->d_ents, p->d_status, p->d_inflate_list, G.h1, sgg, p->d_fb_list, p->d_counter + 52, G.h0);
		int per_sm2 = 0;
		CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm2, k_inflate_lz<OTZ_SEG_RING, false, true>, 128, 4 * sizeof(I2LzSmem<OTZ_SEG_RING>)));
		const uint32_t lgrid = std::max(1u, std::min((uint32_t)(c->sm_count * std::max(per_sm2, 1)), (ng + 3) / 4));
		k_inflate_lz<OTZ_SEG_RING, false, true><<<lgrid, 128, 4 * sizeof(I2LzSmem<OTZ_SEG_RING>), G.st>>>(d_out, p->d_ents, p->d_inflate_list, G.h1,
			p->d_counter + G.c_seglz, c->d_tok_cache, p->d_tok_ofs, p->d_tokres, p->d_status, p->d_produced, sgg, G.h0);
		c->launches += 2;
		if (itrace) {
			CK(cudaEventRecord(tev[4 + g], G.st));
		}
		if (sg.sym_cap) {
			int rc_ = c->seg_ring == 8192 ? launch_seg_par<8192>(c, p, d_out, sgg, G.st, G.h0, G.h1, p->d_counter + G.c_par, p->d_counter + G.c_tr)
			                              : launch_seg_par<4096>(c, p, d_out, sgg, G.st, G.h0, G.h1, p->d_counter + G.c_par, p->d_counter + G.c_tr);
			if (rc_) {
				return rc_;
			}
		}
		CK(cudaGetLastError());
		CK(cudaEventRecord(G.join, G.st));
		if (itrace) {
			CK(cudaEventRecord(tev[7 + g], G.st));
		}
		forked = true;
	}
	if (itrace) {
		CK(cudaEventRecord(tev[10], s));   // (regular streams: tokenizer done)
	}
	if (count) {
		int rc;
		switch (c->lz_ring) {
		case 8192: rc = launch_lz<8192>(c, p, d_out, nh, count, s); break;
		case 16384: rc = launch_lz<16384>(c, p, d_out, nh, count, s); break;
		default: rc = launch_lz<4096>(c, p, d_out, nh, count, s); break;
		}
		if (rc) {
			return rc;
		}
	}
	if (itrace) {
		CK(cudaEventRecord(tev[11], s));   // (regular streams: executed)
	}
	if (forked) {
		for (uint32_t g = 0; g < n_grp; g++) {
			CK(cudaStreamWaitEvent(s, grp[g].join, 0));   // (k_seg_stitch appends to the same fallback list)
		}
	}
	if (itrace) {
		CK(cudaStreamSynchronize(s));
		auto at = [&](int i) {
			float t = 0;
			cudaEventElapsedTime(&t, tev[0], tev[i]);
			return t;
		};
		fprintf(stderr, "otz inflate: %u regular streams: tokenizer done %.2f ms, executed %.2f ms |", count, at(10), at(11));
		for (uint32_t g = 0; g < n_grp; g++) {
			fprintf(stderr, " group %u (%u huge streams): tokenizer %.2f, stitch + walk %.2f, segments / window / translate %.2f ms |", g, grp[g].h1 - grp[g].h0,
				at(1 + g), at(4 + g), at(7 + g));
		}
		fprintf(stderr, "\n");
		for (int i = 0; i < 12; i++) {
			cudaEventDestroy(tev[i]);
		}
	}
	return launch_inflate_cfg(c, p, d_archive, d_out, 32, 4096, 0, p->n_inflate, 16, s, p->d_fb_list, p->d_counter + 52);
}

static int dispatch_inflate(otz_ctx *c, otz_plan *p, const uint8_t *d_archive, uint8_t *d_out) {
	if (c->inflate_mode != 1 && !c->inflate_tile && !c->inflate_ring) {
		// token scratch: grow-only, shared by the runs of this context (they are ordered on its stream)
		if (p->tok_bytes + 64 > c->tok_cache_bytes) {
			CK(cudaStreamSynchronize(c->stream));
			cudaFree(c->d_tok_cache);
			c->d_tok_cache = nullptr;
			c->tok_cache_bytes = 0;
			if (cudaMalloc(&c->d_tok_cache, p->tok_bytes + 64) == cudaSuccess) {
				c->tok_cache_bytes = p->tok_bytes + 64;
			} else {
				cudaGetLastError();   // not enough memory for the token scratch: the one-kernel decoder needs none
			}
		}
		if (c->d_tok_cache) {
			return dispatch_inflate3(c, p, d_archive, d_out);
		}
	}
	if (c->inflate_tile || c->inflate_ring) {   // explicit configuration (tests, sweeps): one kernel for everything
		const int g = c->inflate_tile ? c->inflate_tile : 32;
		const int w = c->inflate_ring ? c->inflate_ring : 2048;
		return launch_inflate_cfg(c, p, d_archive, d_out, g, w, 0, p->n_inflate, 0, c->stream);
	}
	const uint32_t n_big = p->n_inflate_big, n_small = p->n_inflate - n_big;
	const bool small_big_ring = n_small <= (uint32_t)c->sm_count * 10u;
	int rc = OTZ_SUCCESS;
	if (n_big && n_small && !small_big_ring) {
		CK(cudaEventRecord(c->ev_fork, c->stream));
		CK(cudaStreamWaitEvent(c->stream2, c->ev_fork, 0));
		rc = launch_inflate_cfg(c, p, d_archive, d_out, 32, 16384, 0, n_big, 0, c->stream2);
		if (rc) {
			return rc;
		}
		rc = launch_inflate_cfg(c, p, d_archive, d_out, 32, 2048, n_big, n_small, 16, c->stream);
		CK(cudaEventRecord(c->ev_join, c->stream2));
		CK(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
		return rc;
	}
	if (small_big_ring) {
		return launch_inflate_cfg(c, p, d_archive, d_out, 32, 16384, 0, p->n_inflate, 0, c->stream);
	}
	return launch_inflate_cfg(c, p, d_archive, d_out, 32, 2048, 0, p->n_inflate, 0, c->stream);
}

// Deflate64 entries (k_inflate<G, W, true>): launched right behind k_resolve on streams of their own, so that they run next to
// the DEFLATE and Zstandard work of the run; *joins = number of ev_d64_join events the main stream must wait for before the
// CRC.  The launches are sized as dispatch_inflate's legacy branch sizes them; OTZ_INFLATE_TILE / OTZ_INFLATE_RING select one
// instantiation for all of them.  Work counters: words 24 and 25 of d_counter, which no other launch uses.
static int dispatch_deflate64(otz_ctx *c, otz_plan *p, const uint8_t *d_archive, uint8_t *d_out, int *joins) {
	CK(cudaEventRecord(c->ev_d64_fork, c->stream));
	int &used = *joins, rc = OTZ_SUCCESS;
	used = 0;
	auto launch = [&](int g, int w, uint32_t first, uint32_t count) {
		cudaStream_t st = c->stream_d64[used];
		CK(cudaStreamWaitEvent(st, c->ev_d64_fork, 0));
		const int r = launch_inflate_cfg<true>(c, p, d_archive, d_out, g, w, first, count, 24 + used, st);
		CK(cudaEventRecord(c->ev_d64_join[used], st));
		used++;
		return r;
	};
	const uint32_t n_big = p->n_d64_big, n_small = p->n_d64 - n_big;
	if (c->inflate_tile || c->inflate_ring) {
		rc = launch(c->inflate_tile ? c->inflate_tile : 32, c->inflate_ring ? c->inflate_ring : 2048, 0, p->n_d64);
	} else if (n_small <= (uint32_t)c->sm_count * 10u) {
		rc = launch(32, 16384, 0, p->n_d64);
	} else {
		if (n_big) {
			rc = launch(32, 16384, 0, n_big);
		}
		if (rc == OTZ_SUCCESS) {
			rc = launch(32, 2048, n_big, n_small);
		}
	}
	return rc;
}

template <int LCLP>
static int launch_lzma(otz_ctx *c, otz_plan *p, const uint8_t *d_archive, uint8_t *d_out, uint32_t *d_work, const uint32_t *d_n_class) {
	const size_t smem = sizeof(XzSmem<LCLP>);
	int per_sm = 0;
	CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_lzma<LCLP>, 32, smem));
	const uint32_t grid = std::max(1u, std::min((uint32_t)(c->sm_count * std::max(per_sm, 1)), p->n_xz_slots));
	k_lzma<LCLP><<<grid, 32, smem, c->stream_xz>>>(d_archive, d_out, p->d_ents, p->d_est, p->d_xz_list, p->d_xz_ent, p->d_xz_segs,
		p->n_xz_slots, d_work, d_n_class);
	c->launches++;
	CK(cudaGetLastError());
	return OTZ_SUCCESS;
}

// XZ entries (k_xz.cuh): walk, decode (one launch per shared-memory class) and verdicts on a stream of their own, forked
// behind k_resolve and joined before the CRC.  Words of d_counter: 26 / 27 = slot counters of the two k_lzma launches,
// 28 / 29 = segments of each class (counted by the walk; a launch whose class has none returns at once).
static int dispatch_xz(otz_ctx *c, otz_plan *p, const uint8_t *d_archive, uint8_t *d_out) {
	cudaStream_t st = c->stream_xz;
	CK(cudaEventRecord(c->ev_xz_fork, c->stream));
	CK(cudaStreamWaitEvent(st, c->ev_xz_fork, 0));
	const uint32_t *t0 = reinterpret_cast<const uint32_t *>(reinterpret_cast<const uint8_t *>(c->d_tabs) + offsetof(OtzCrcTables, t0));
	k_xz_walk<<<(p->n_xz + 127) / 128, 128, 0, st>>>(d_archive, p->d_ents, p->d_est, p->d_status, p->d_xz_list, p->n_xz, p->d_xz_ent,
		p->d_xz_segs, t0, p->d_counter + 28);
	c->launches++;
	int rc = launch_lzma<3>(c, p, d_archive, d_out, p->d_counter + 26, p->d_counter + 28);
	if (rc == OTZ_SUCCESS) {
		rc = launch_lzma<4>(c, p, d_archive, d_out, p->d_counter + 27, p->d_counter + 29);
	}
	if (rc) {
		return rc;
	}
	k_xz_finish<<<(p->n_xz + 7) / 8, 256, 0, st>>>(d_out, p->d_ents, p->d_status, p->d_produced, p->d_xz_list, p->n_xz, p->d_xz_ent,
		p->d_xz_segs);
	c->launches++;
	CK(cudaEventRecord(c->ev_xz_join, st));
	return OTZ_SUCCESS;
}

extern "C" int otz_extract_run(otz_ctx *c, otz_plan *p, const uint8_t *d_archive, uint64_t archive_len, uint8_t *d_out,
	uint64_t out_len) {
	if (!c || !p || (!d_archive && archive_len)) {
		return OTZ_ERR_ARG;
	}
	if (p->out_bytes_needed > out_len || (p->out_bytes_needed && !d_out)) {
		snprintf(g_err, sizeof(g_err), "output arena too small: need %llu, have %llu", (unsigned long long)p->out_bytes_needed,
			(unsigned long long)out_len);
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	cudaStream_t s = c->stream;
	const uint32_t n = p->n;
	cudaEvent_t *pev = c->pev[c->prof_runs % OTZ_PROF_SLOTS];
	if (c->profile) {
		CK(cudaEventRecord(pev[0], s));
	}
	if (n) {
		CK(cudaMemsetAsync(p->d_counter, 0, 256, s));
		k_resolve<<<(n + 255) / 256, 256, 0, s>>>(d_archive, archive_len, out_len, p->d_ents, n, p->d_est, p->d_status, p->d_acc, p->d_produced,
			p->opts);
		c->launches++;
	}
	if (c->profile) {
		CK(cudaEventRecord(pev[1], s));
	}
	int d64_joins = 0;
	if (p->n_d64) {
		const int rc = dispatch_deflate64(c, p, d_archive, d_out, &d64_joins);
		if (rc) {
			return rc;
		}
	}
	if (p->n_xz) {
		const int rc = dispatch_xz(c, p, d_archive, d_out);
		if (rc) {
			return rc;
		}
	}
	if (p->n_store_chunks && !p->opts.verify_only) {
		k_store_copy<<<std::min((uint32_t)c->sm_count * 4, (p->n_store_chunks + 7) / 8), 256, 0, s>>>(d_archive, d_out, p->d_ents, p->d_est,
			p->d_status, p->d_chunks, p->n_store_chunks);
		c->launches++;
	}
	if (p->n_zstd) {
		k_zstdref<<<std::min((uint32_t)c->sm_count * 4, (p->n_zstd + 7) / 8), 256, 0, s>>>(d_archive, d_out, p->d_ents, p->d_est, p->d_status,
			p->d_zstd_list, p->n_zstd);
		c->launches++;
		// entries that are not a reference container but carry the Zstandard magic: RFC 8878 frames, decoded in two
		// phases (literal / sequence tokenizers + the LZ executor of the inflate path) over the context's token scratch
		if (p->ztok_bytes + 64 > c->ztok_cache_bytes) {
			CK(cudaStreamSynchronize(c->stream));
			cudaFree(c->d_ztok_cache);
			c->d_ztok_cache = nullptr;
			c->ztok_cache_bytes = 0;
			if (cudaMalloc(&c->d_ztok_cache, p->ztok_bytes + 64) != cudaSuccess) {
				return fail_cuda(cudaGetLastError(), "cudaMalloc(Zstandard token scratch)");
			}
			c->ztok_cache_bytes = p->ztok_bytes + 64;
		}
		{
			static bool zattr2 = false;
			const int zsmem2 = (int)(ZS_LIT_WARPS * 8 * sizeof(ZsLitSmem));
			if (!zattr2) {
				CK(cudaFuncSetAttribute(k_zstd_lit, cudaFuncAttributeMaxDynamicSharedMemorySize, zsmem2));
				CK(cudaFuncSetAttribute(k_zstd_seq, cudaFuncAttributeMaxDynamicSharedMemorySize, ZS_SEQ_WARPS * ZS_SEQ_LPW_MAX * ZS_SEQ_TAB_BYTES));
				CK(cudaFuncSetAttribute(k_inflate_lz<4096, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(4 * sizeof(I2LzSmem<4096>))));
				zattr2 = true;
			}
			uint32_t *const litres = reinterpret_cast<uint32_t *>(p->d_ztokres + p->n_zstd);
			// OTZ_ZSTD_TRACE=1: durations of the three kernels of this path, printed to stderr (a diagnostic: it waits for them)
			const bool ztrace = getenv("OTZ_ZSTD_TRACE") != nullptr;
			cudaEvent_t zev[4] = { nullptr, nullptr, nullptr, nullptr };
			if (ztrace) {
				for (int i = 0; i < 4; i++) {
					CK(cudaEventCreate(&zev[i]));
				}
				CK(cudaEventRecord(zev[0], s));
			}
			uint32_t *const seqres = litres + p->n_zstd;
			int per_sm = 0;
			// sequences on the main stream FIRST (one CTA of ZS_SEQ_WARPS warps per SM, as many lanes per warp as the batch needs:
			// their tables are the shared memory), literals on a side stream next to them: the CTAs of the literal kernel take the
			// shared memory and the issue slots the sequence kernel leaves
			const uint32_t zw = ZS_SEQ_WARPS;
			const uint32_t zlpw = std::max(1u, std::min((uint32_t)ZS_SEQ_LPW_MAX, (p->n_zstd + c->sm_count * zw - 1) / (c->sm_count * zw)));
			const uint32_t sgrid = std::max(1u, std::min((uint32_t)c->sm_count, (p->n_zstd + zlpw * zw - 1) / (zlpw * zw)));
			CK(cudaEventRecord(c->ev_fork, s));
			k_zstd_seq<<<sgrid, 32 * zw, zw * zlpw * ZS_SEQ_TAB_BYTES, s>>>(d_archive, p->d_ents, p->d_est, p->d_status, p->d_zstd_list,
				p->n_zstd, c->d_ztok_cache, p->d_ztok_ofs, p->d_ztokres, seqres, p->d_counter + 34, zlpw);
			c->launches++;
			if (ztrace) {
				CK(cudaEventRecord(zev[1], s));
			}
			CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_zstd_lit, 32 * ZS_LIT_WARPS, zsmem2));
			const uint32_t zgrid = std::max(1u, std::min((uint32_t)(c->sm_count * std::max(per_sm, 1)), (p->n_zstd + 8 * ZS_LIT_WARPS - 1) / (8 * ZS_LIT_WARPS)));
			CK(cudaStreamWaitEvent(c->stream4, c->ev_fork, 0));
			k_zstd_lit<<<zgrid, 32 * ZS_LIT_WARPS, zsmem2, c->stream4>>>(d_archive, p->d_ents, p->d_est, p->d_status, p->d_zstd_list, p->n_zstd, c->d_ztok_cache,
				p->d_ztok_ofs, litres, p->d_counter + 32);
			c->launches++;
			CK(cudaEventRecord(c->ev_join4, c->stream4));
			CK(cudaStreamWaitEvent(s, c->ev_join4, 0));
			k_zstd_join<<<(p->n_zstd + 255) / 256, 256, 0, s>>>(p->d_zstd_list, p->n_zstd, litres, seqres, p->d_ztokres, p->d_status);
			c->launches++;
			if (ztrace) {
				CK(cudaEventRecord(zev[2], s));
			}
			CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_inflate_lz<4096, true, false>, 128, 4 * sizeof(I2LzSmem<4096>)));
			const uint32_t lgrid = std::max(1u, std::min((uint32_t)(c->sm_count * std::max(per_sm, 1)), (p->n_zstd + 3) / 4));
			k_inflate_lz<4096, true, false><<<lgrid, 128, 4 * sizeof(I2LzSmem<4096>), s>>>(d_out, p->d_ents, p->d_zstd_list, p->n_zstd, p->d_counter + 36,
				c->d_ztok_cache, p->d_ztok_ofs, p->d_ztokres, p->d_status, p->d_produced, I2SegCtl{}, 0u);
			c->launches++;
			if (ztrace) {
				CK(cudaEventRecord(zev[3], s));
				CK(cudaEventSynchronize(zev[3]));
				float t[3];
				for (int i = 0; i < 3; i++) {
					CK(cudaEventElapsedTime(&t[i], zev[i], zev[i + 1]));
				}
				fprintf(stderr, "otz zstd: %u entries | k_zstd_seq %.3f ms (grid %u, %u lanes per warp)  + k_zstd_lit on a side stream (grid %u) + join %.3f ms  k_inflate_lz<wide> %.3f ms\n",
					p->n_zstd, t[0], sgrid, zlpw, zgrid, t[1], t[2]);
				for (int i = 0; i < 4; i++) {
					cudaEventDestroy(zev[i]);
				}
			}
		}
	}
	if (p->n_inflate) {
		int rc = dispatch_inflate(c, p, d_archive, d_out);
		if (rc) {
			return rc;
		}
	}
	for (int k = 0; k < d64_joins; k++) {
		CK(cudaStreamWaitEvent(s, c->ev_d64_join[k], 0));
	}
	if (p->n_xz) {
		CK(cudaStreamWaitEvent(s, c->ev_xz_join, 0));
	}
	if (c->profile) {
		CK(cudaEventRecord(pev[2], s));
	}
	// every chunk: STORE payloads in place when verify_only, else from the arena
	const uint32_t crc_first = 0u;
	if (p->n_chunks > crc_first) {
		// persistent: exactly the resident CTAs (register-limited), each striding over the chunk list
		const uint32_t nc = p->n_chunks - crc_first;
		const uint32_t grid = std::min((uint32_t)c->sm_count * crc_ctas_per_sm(), (nc + 7) / 8);
		k_crc_chunks<<<grid, 256, 0, s>>>(d_archive, d_out, p->d_ents, p->d_est, p->d_status, p->d_chunks + crc_first, nc, p->d_acc, c->d_tabs,
			p->opts.verify_only, 0);
		c->launches++;
	}
	if (p->n_zchunks) {
		const uint32_t grid = std::min((uint32_t)c->sm_count * crc_ctas_per_sm(), (p->n_zchunks + 7) / 8);
		k_crc_chunks<<<grid, 256, 0, s>>>(d_archive, d_out, p->d_ents, p->d_est, p->d_status, p->d_zchunks, p->n_zchunks, p->d_acc, c->d_tabs, 0, 0);
		c->launches++;
	}
	if (c->profile) {
		CK(cudaEventRecord(pev[3], s));
	}
	if (n) {
		k_crc_finalize<<<(n + 255) / 256, 256, 0, s>>>(p->d_ents, n, p->d_acc, p->d_crc, p->d_status, c->d_tabs);
		c->launches++;
	}
	if (c->profile) {
		CK(cudaEventRecord(pev[4], s));
		c->prof_runs++;
	}
	CK(cudaGetLastError());
	return OTZ_SUCCESS;
}

extern "C" int otz_extract_results(otz_ctx *c, otz_plan *p, uint32_t *crc, int32_t *status) {
	if (!c || !p) {
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	if (p->n && crc) {
		CK(cudaMemcpyAsync(crc, p->d_crc, p->n * 4ull, cudaMemcpyDeviceToHost, c->stream));
	}
	if (p->n && status) {
		CK(cudaMemcpyAsync(status, p->d_status, p->n * 4ull, cudaMemcpyDeviceToHost, c->stream));
	}
	CK(cudaMemcpyAsync(&c->last_fallbacks, p->d_counter + 52, 4, cudaMemcpyDeviceToHost, c->stream));
	CK(cudaStreamSynchronize(c->stream));
	return OTZ_SUCCESS;
}

extern "C" uint32_t otz_inflate_fallbacks(otz_ctx *c) { return c ? c->last_fallbacks : 0; }

extern "C" int otz_extract_produced(otz_ctx *c, otz_plan *p, uint32_t *produced) {
	if (!c || !p || !produced) {
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	if (p->n) {
		CK(cudaMemcpyAsync(produced, p->d_produced, p->n * 4ull, cudaMemcpyDeviceToHost, c->stream));
	}
	CK(cudaStreamSynchronize(c->stream));
	return OTZ_SUCCESS;
}

extern "C" int otz_extract_host(otz_ctx *c, const uint8_t *archive, uint64_t archive_len, const otz_entry *ents, uint32_t n,
	const otz_extract_opts *opts, uint8_t *out, uint64_t out_len, uint32_t *crc, int32_t *status) {
	return otz_extract_host_ex(c, archive, archive_len, ents, n, opts, out, out_len, crc, status, nullptr);
}

// Grow-only scratch of a context (token scratch of the two-phase decoders, symbol buffer of the parallel segment execution) for
// the plan about to run: the pipelined host call reserves it before anything is in flight, so that no cudaFree / cudaMalloc
// (which synchronise the device) lands between its asynchronous stages.  Failing to allocate is not an error here: the
// dispatchers fall back to the decoders that need no scratch.
static int reserve_scratch(otz_ctx *c, otz_plan *p) {
	if (p->n_inflate) {
		const int rc_ = reserve_spec_tmp(c);
		if (rc_) {
			return rc_;
		}
	}
	if (p->n_inflate && p->tok_bytes + 64 > c->tok_cache_bytes) {
		CK(cudaStreamSynchronize(c->stream));
		cudaFree(c->d_tok_cache);
		c->d_tok_cache = nullptr;
		c->tok_cache_bytes = 0;
		if (cudaMalloc(&c->d_tok_cache, p->tok_bytes + 64) == cudaSuccess) {
			c->tok_cache_bytes = p->tok_bytes + 64;
		} else {
			cudaGetLastError();
		}
	}
	if (p->n_zstd && p->ztok_bytes + 64 > c->ztok_cache_bytes) {
		CK(cudaStreamSynchronize(c->stream));
		cudaFree(c->d_ztok_cache);
		c->d_ztok_cache = nullptr;
		c->ztok_cache_bytes = 0;
		if (cudaMalloc(&c->d_ztok_cache, p->ztok_bytes + 64) == cudaSuccess) {
			c->ztok_cache_bytes = p->ztok_bytes + 64;
		} else {
			cudaGetLastError();
		}
	}
	if (p->sym_elems > c->sym_cache_elems && !c->seg_serial) {
		CK(cudaStreamSynchronize(c->stream));
		CK(cudaStreamSynchronize(c->stream2));
		cudaFree(c->d_sym_cache);
		c->d_sym_cache = nullptr;
		c->sym_cache_elems = 0;
		if (cudaMalloc(&c->d_sym_cache, p->sym_elems * 2 + 64) == cudaSuccess) {
			c->sym_cache_elems = p->sym_elems;
		} else {
			cudaGetLastError();
		}
	}
	return OTZ_SUCCESS;
}

// One sub-batch of the pipelined host call: a contiguous index range of the caller's table with its byte range of the
// archive image and of the output arena.
struct OtzSub {
	uint32_t first, n;
	uint64_t a_lo, a_hi;   // archive bytes [a_lo, a_hi) hold every LFH and payload of the range
	uint64_t o_lo, o_hi;   // arena bytes the range writes
	otz_plan *plan;
};

// Byte range of entry e in the host image: LFH + name + extra + payload (clamped to the image; the kernels re-check
// everything on the device, this only decides what is uploaded).
static void entry_span(const uint8_t *archive, uint64_t archive_len, const otz_entry &e, uint64_t *lo, uint64_t *hi) {
	uint64_t b = std::min<uint64_t>(e.lfh_ofs, archive_len), t = b;
	if (e.flags & OTZ_EF_CHUNK) {
		t = b + e.comp_size;   // chunk rows address their payload directly
	} else if (archive_len - b >= 30) {
		const uint64_t nl = archive[b + 26] | (archive[b + 27] << 8), xl = archive[b + 28] | (archive[b + 29] << 8);
		t = b + 30 + nl + xl + e.comp_size;
	} else {
		t = archive_len;
	}
	*lo = b & ~63ull;
	*hi = std::min<uint64_t>(archive_len, (t + 63) & ~63ull);
}

extern "C" int otz_extract_host_ex(otz_ctx *c, const uint8_t *archive, uint64_t archive_len, const otz_entry *ents, uint32_t n,
	const otz_extract_opts *opts, uint8_t *out, uint64_t out_len, uint32_t *crc, int32_t *status, uint32_t *produced) {
	if (!c || !opts || (n && !ents) || (archive_len && !archive)) {
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	// ---- sub-batches: contiguous index ranges of ~OTZ_PIPE_BYTES of output whose archive ranges ascend without overlap
	// (true for every archive laid out in index order).  Two lanes (child contexts: own streams and scratch) alternate,
	// so H2D(k+1), the kernels of k and D2H(k-1) overlap.  Tables with chunk rows (their parent links are table
	// indices) or out-of-order payloads go as one batch.
	// (few, large sub-batches: the kernels of a batch lose efficiency when its largest stream becomes their critical path,
	// while the copies — the bound of the whole call — do not care; twelve keep the ramp, H2D + kernels of the first one, at
	// a few percent of the copy time)
	const char *pb = getenv("OTZ_PIPE_BYTES");
	uint64_t target = pb ? strtoull(pb, nullptr, 0) : (256ull << 20);
	if (!pb) {
		uint64_t total = 0;
		for (uint32_t i = 0; i < n; i++) {
			total += (uint64_t)ents[i].uncomp_size + ents[i].comp_size;
		}
		target = std::max<uint64_t>(target, total / 12 + 1);
	}
	std::vector<OtzSub> subs;
	bool pipelined = target != 0 && n > 1;
	uint64_t need = 0;
	for (uint32_t i = 0; i < n; i++) {
		if (ents[i].flags & (OTZ_EF_CHUNK | OTZ_EF_PARENT)) {
			pipelined = false;
		}
		if (!(opts->verify_only && ents[i].method == OTZ_M_STORE)) {
			need = std::max<uint64_t>(need, ents[i].out_ofs + ents[i].uncomp_size);
		}
	}
	if (need > out_len || (need && !out && !opts->verify_only)) {
		snprintf(g_err, sizeof(g_err), "output arena too small: need %llu, have %llu", (unsigned long long)need, (unsigned long long)out_len);
		return OTZ_ERR_ARG;
	}
	if (pipelined) {
		OtzSub cur = { 0, 0, ~0ull, 0, ~0ull, 0, nullptr };
		uint64_t bytes = 0, prev_a_hi = 0, prev_o_hi = 0;
		for (uint32_t i = 0; i < n && pipelined; i++) {
			uint64_t lo, hi;
			entry_span(archive, archive_len, ents[i], &lo, &hi);
			const bool writes = !(opts->verify_only && ents[i].method == OTZ_M_STORE);
			const uint64_t olo = writes ? ents[i].out_ofs : ~0ull, ohi = writes ? ents[i].out_ofs + ents[i].uncomp_size : 0;
			cur.a_lo = std::min(cur.a_lo, lo);
			cur.a_hi = std::max(cur.a_hi, hi);
			cur.o_lo = std::min(cur.o_lo, olo);
			cur.o_hi = std::max(cur.o_hi, ohi);
			cur.n++;
			bytes += (uint64_t)ents[i].uncomp_size + ents[i].comp_size;
			// (ramp: the first two sub-batches are a quarter and a half of the rest, so that the D2H stream — the bound of the
			// call — starts after a quarter of a sub-batch's H2D + kernels instead of a whole one)
			const uint64_t tgt = subs.size() == 0 ? target / 4 : subs.size() == 1 ? target / 2 : target;
			if (bytes >= tgt || i + 1 == n) {
				// (ranges are 64-byte aligned: neighbours may share their boundary block, which then is copied twice with the same bytes —
				// only real overlap, payloads out of index order, turns the pipeline off)
				if (cur.a_lo + 64 < prev_a_hi || (cur.o_hi > cur.o_lo && cur.o_lo < prev_o_hi)) {
					pipelined = false;
					break;
				}
				prev_a_hi = cur.a_hi;
				prev_o_hi = std::max(prev_o_hi, cur.o_hi);
				subs.push_back(cur);
				cur = OtzSub{ i + 1, 0, ~0ull, 0, ~0ull, 0, nullptr };
				bytes = 0;
			}
		}
		if (subs.size() < 2) {
			pipelined = false;
		}
	}
	// device staging buffers are kept (grow-only) so repeated calls pay only for the copies
	int rc = OTZ_SUCCESS;
	if (archive_len > c->arch_cache_bytes || !c->d_arch_cache) {
		cudaFree(c->d_arch_cache);
		c->d_arch_cache = nullptr;
		c->arch_cache_bytes = 0;
		if ((rc = otz_dev_alloc(c, archive_len, &c->d_arch_cache))) {
			return rc;
		}
		c->arch_cache_bytes = archive_len;
	}
	if (need > c->out_cache_bytes) {
		cudaFree(c->d_out_cache);
		c->d_out_cache = nullptr;
		c->out_cache_bytes = 0;
		if ((rc = otz_dev_alloc(c, need, &c->d_out_cache))) {
			return rc;
		}
		c->out_cache_bytes = need;
	}
	const uint8_t *d_arch = (const uint8_t *)c->d_arch_cache;
	uint8_t *d_out = (uint8_t *)c->d_out_cache;
	if (!pipelined) {
		otz_plan *p = nullptr;
		if ((rc = otz_plan_create(c, ents, n, opts, &p))) {
			return rc;
		}
		do {
			// only the bytes the entries of this call live in (a window of a large archive uploads its own range)
			uint64_t lo = archive_len, hi = 0;
			for (uint32_t i = 0; i < n; i++) {
				uint64_t a, b;
				entry_span(archive, archive_len, ents[i], &a, &b);
				lo = std::min(lo, a);
				hi = std::max(hi, b);
			}
			if (hi > lo && (rc = otz_h2d(c, (uint8_t *)c->d_arch_cache + lo, archive + lo, hi - lo))) break;
			if ((rc = otz_extract_run(c, p, d_arch, archive_len, d_out, need))) break;
			if (out && need && (rc = otz_d2h(c, out, c->d_out_cache, need))) break;
			rc = otz_extract_results(c, p, crc, status);
			if (!rc && produced) {
				rc = otz_extract_produced(c, p, produced);
			}
		} while (0);
		cudaStreamSynchronize(c->stream);
		otz_plan_destroy(c, p);
		return rc;
	}
	// ---- pipelined
	for (int l = 0; l < 2; l++) {
		if (!c->pipe[l] && (rc = otz_ctx_create(c->device, &c->pipe[l]))) {
			return rc;
		}
	}
	// pinned staging for the per-entry results (a D2H copy into pageable memory would block the enqueueing thread)
	const uint64_t res_bytes = (uint64_t)n * 12 + subs.size() * 4 + 64;
	if (res_bytes > c->h_res_bytes) {
		cudaFreeHost(c->h_res);
		c->h_res = nullptr;
		c->h_res_bytes = 0;
		if (cudaHostAlloc(&c->h_res, res_bytes, cudaHostAllocDefault) != cudaSuccess) {
			return fail_cuda(cudaGetLastError(), "cudaHostAlloc(result staging)");
		}
		c->h_res_bytes = res_bytes;
	}
	uint32_t *h_crc = (uint32_t *)c->h_res, *h_prod = h_crc + n, *h_fb = h_prod + n + n;
	int32_t *h_st = (int32_t *)(h_prod + n);
	// the sub-plans (work lists, device tables: ~30 allocations each) of the last pipelined call are kept: a caller that
	// extracts the same table again (same rows, same options) pays for the copies and the kernels only
	const bool cached = c->pc_n == n && c->pc_plans.size() == subs.size() && !memcmp(&c->pc_opts, opts, sizeof(*opts)) &&
		(n == 0 || !memcmp(c->pc_ents.data(), ents, (size_t)n * sizeof(otz_entry)));
	if (!cached) {
		for (size_t k = 0; k < c->pc_plans.size(); k++) {
			otz_plan_destroy(c->pipe[k & 1], c->pc_plans[k]);
		}
		c->pc_plans.clear();
		c->pc_n = 0;
	}
	for (auto &sb : subs) {   // all plans first: cudaMalloc / cudaFree must not sit between the asynchronous stages
		const size_t k = &sb - &subs[0];
		if (cached) {
			sb.plan = c->pc_plans[k];
			continue;
		}
		if ((rc = otz_plan_create(c->pipe[k & 1], ents + sb.first, sb.n, opts, &sb.plan))) {
			break;
		}
	}
	if (!rc) {
		// scratch of both lanes, sized for their largest sub-batch, before anything is in flight
		for (auto &sb : subs) {
			otz_ctx *lc = c->pipe[(&sb - &subs[0]) & 1];
			if ((rc = reserve_scratch(lc, sb.plan))) {
				break;
			}
		}
	}
	// OTZ_PIPE_TRACE=1: event timestamps of every stage, printed to stderr after the call (evidence for the overlap)
	const bool trace = getenv("OTZ_PIPE_TRACE") != nullptr;
	std::vector<cudaEvent_t> tev;
	if (trace) {
		tev.resize(subs.size() * 4);
		for (auto &e : tev) {
			cudaEventCreate(&e);
		}
	}
	for (size_t k = 0; k < subs.size() && !rc; k++) {
		OtzSub &sb = subs[k];
		otz_ctx *lc = c->pipe[k & 1];
		cudaStream_t st = lc->stream;
		if (trace) {
			cudaEventRecord(tev[4 * k], st);
		}
		if (sb.a_hi > sb.a_lo) {
			CK(cudaMemcpyAsync((uint8_t *)c->d_arch_cache + sb.a_lo, archive + sb.a_lo, sb.a_hi - sb.a_lo, cudaMemcpyHostToDevice, st));
		}
		if (trace) {
			cudaEventRecord(tev[4 * k + 1], st);
		}
		if ((rc = otz_extract_run(lc, sb.plan, d_arch, archive_len, d_out, need))) {
			break;
		}
		if (trace) {
			cudaEventRecord(tev[4 * k + 2], st);
		}
		if (out && sb.o_hi > sb.o_lo) {
			CK(cudaMemcpyAsync(out + sb.o_lo, d_out + sb.o_lo, sb.o_hi - sb.o_lo, cudaMemcpyDeviceToHost, st));
		}
		if (trace) {
			cudaEventRecord(tev[4 * k + 3], st);
		}
		CK(cudaMemcpyAsync(h_crc + sb.first, sb.plan->d_crc, sb.n * 4ull, cudaMemcpyDeviceToHost, st));
		CK(cudaMemcpyAsync(h_st + sb.first, sb.plan->d_status, sb.n * 4ull, cudaMemcpyDeviceToHost, st));
		CK(cudaMemcpyAsync(h_prod + sb.first, sb.plan->d_produced, sb.n * 4ull, cudaMemcpyDeviceToHost, st));
		CK(cudaMemcpyAsync(h_fb + k, sb.plan->d_counter + 52, 4, cudaMemcpyDeviceToHost, st));
	}
	for (int l = 0; l < 2; l++) {
		cudaError_t e = cudaStreamSynchronize(c->pipe[l]->stream);
		if (e != cudaSuccess && !rc) {
			rc = fail_cuda(e, "pipelined extract");
		}
	}
	if (trace) {
		for (size_t k = 0; k < subs.size() && !rc; k++) {
			float t[4];
			for (int j = 0; j < 4; j++) {
				cudaEventElapsedTime(&t[j], tev[0], tev[4 * k + j]);
			}
			fprintf(stderr, "otz pipe: sub %2zu lane %zu rows %6u  in %7.1f MB out %8.1f MB | start %7.2f  h2d-done %7.2f  kernels-done %7.2f  d2h-done %7.2f ms\n", k, k & 1,
				subs[k].n, (subs[k].a_hi - subs[k].a_lo) / 1e6, (subs[k].o_hi > subs[k].o_lo ? subs[k].o_hi - subs[k].o_lo : 0) / 1e6, t[0], t[1], t[2], t[3]);
		}
		for (auto &e : tev) {
			cudaEventDestroy(e);
		}
	}
	if (!rc) {
		if (crc) {
			memcpy(crc, h_crc, n * 4ull);
		}
		if (status) {
			memcpy(status, h_st, n * 4ull);
		}
		if (produced) {
			memcpy(produced, h_prod, n * 4ull);
		}
		c->last_fallbacks = 0;
		for (size_t k = 0; k < subs.size(); k++) {
			c->last_fallbacks += h_fb[k];
		}
	}
	uint64_t child_launches = 0;
	if (!rc) {
		if (!cached) {
			c->pc_plans.clear();
			for (auto &sb : subs) {
				c->pc_plans.push_back(sb.plan);
			}
			c->pc_ents.assign(ents, ents + n);
			c->pc_opts = *opts;
			c->pc_n = n;
		}
	} else {
		for (auto &sb : subs) {
			otz_plan_destroy(c->pipe[(&sb - &subs[0]) & 1], sb.plan);
		}
		c->pc_plans.clear();
		c->pc_n = 0;
	}
	for (int l = 0; l < 2; l++) {
		child_launches += c->pipe[l]->launches;
		c->pipe[l]->launches = 0;
	}
	c->launches += child_launches;
	return rc;
}

// Multi-GPU host call (SURVEY.md §8e): entries are independent (otezip.c:399-477), so the table is cut into one contiguous
// index range per device, balanced by comp + uncomp bytes (otz_partition); every device gets ONLY its byte range of the
// archive image and of the arena (the offsets of its rows are rebased), runs the pipelined single-device call on its own
// host thread, and the per-entry results land in the caller's arrays at the rows' positions.  No collective, no peer traffic.
extern "C" int otz_extract_host_multi(otz_ctx *const *ctxs, uint32_t n_ctx, const uint8_t *archive, uint64_t archive_len, const otz_entry *ents,
	uint32_t n, const otz_extract_opts *opts, uint8_t *out, uint64_t out_len, uint32_t *crc, int32_t *status, uint32_t *produced) {
	if (!ctxs || !n_ctx || !ctxs[0] || !opts || (n && !ents)) {
		return OTZ_ERR_ARG;
	}
	bool plain = true;
	for (uint32_t i = 0; i < n; i++) {
		plain = plain && !(ents[i].flags & (OTZ_EF_CHUNK | OTZ_EF_PARENT));   // (chunk rows link to table indices: one device)
	}
	if (n_ctx == 1 || n < 2 * n_ctx || !plain) {
		return otz_extract_host_ex(ctxs[0], archive, archive_len, ents, n, opts, out, out_len, crc, status, produced);
	}
	std::vector<uint32_t> first(n_ctx + 1);
	int rc = otz_partition(ents, n, n_ctx, first.data());
	if (rc) {
		return rc;
	}
	std::vector<int> rcs(n_ctx, OTZ_SUCCESS);
	std::vector<std::string> errs(n_ctx);
	std::vector<std::thread> th;
	for (uint32_t g = 0; g < n_ctx; g++) {
		const uint32_t a = first[g], cnt = first[g + 1] - first[g];
		if (!cnt) {
			continue;
		}
		th.emplace_back([=, &rcs, &errs]() {
			// the part's byte ranges, then its rows rebased onto them
			uint64_t a_lo = archive_len, a_hi = 0, o_lo = ~0ull, o_hi = 0;
			for (uint32_t i = a; i < a + cnt; i++) {
				uint64_t lo, hi;
				entry_span(archive, archive_len, ents[i], &lo, &hi);
				a_lo = std::min(a_lo, std::min<uint64_t>(lo, ents[i].lfh_ofs & ~63ull));
				a_hi = std::max(a_hi, hi);
				if (!(opts->verify_only && ents[i].method == OTZ_M_STORE)) {
					o_lo = std::min<uint64_t>(o_lo, ents[i].out_ofs);   // (exact: the copy back must not touch a neighbour's bytes)
					o_hi = std::max<uint64_t>(o_hi, ents[i].out_ofs + ents[i].uncomp_size);
				}
			}
			if (o_hi <= o_lo) {
				o_lo = o_hi = 0;
			}
			a_hi = std::max(a_hi, a_lo);
			o_hi = std::min(o_hi, out_len);
			std::vector<otz_entry> part(ents + a, ents + a + cnt);
			for (auto &e : part) {
				// (a row whose header lies outside the image keeps an offset beyond the part: k_resolve reports the range error)
				e.lfh_ofs = e.lfh_ofs >= a_lo ? e.lfh_ofs - a_lo : ~0ull;
				e.out_ofs = e.out_ofs >= o_lo ? e.out_ofs - o_lo : ~0ull;
			}
			rcs[g] = otz_extract_host_ex(ctxs[g], archive + a_lo, a_hi - a_lo, part.data(), cnt, opts, out ? out + o_lo : nullptr, o_hi - o_lo, crc ? crc + a : nullptr,
				status ? status + a : nullptr, produced ? produced + a : nullptr);
			if (rcs[g]) {
				errs[g] = g_err;
			}
		});
	}
	for (auto &t : th) {
		t.join();
	}
	uint32_t fb = 0;
	for (uint32_t g = 0; g < n_ctx; g++) {
		if (rcs[g] && !rc) {
			rc = rcs[g];
			snprintf(g_err, sizeof(g_err), "device %u: %s", g, errs[g].c_str());
		}
		fb += ctxs[g]->last_fallbacks;
	}
	ctxs[0]->last_fallbacks = fb;
	return rc;
}

// ---------------------------------------------------------------- multi-GPU sharding (host only)
extern "C" int otz_partition(const otz_entry *ents, uint32_t n, uint32_t parts, uint32_t *first) {
	if (!first || !parts || (n && !ents)) {
		return OTZ_ERR_ARG;
	}
	uint64_t total = 0;
	for (uint32_t i = 0; i < n; i++) {
		total += (uint64_t)ents[i].comp_size + ents[i].uncomp_size + 64u;   // (+ a constant per entry: empty entries cost a table row)
	}
	// boundary g = the first index whose prefix weight reaches g/parts of the total (rounded to the nearer side)
	uint64_t acc = 0;
	uint32_t g = 1;
	first[0] = 0;
	for (uint32_t i = 0; i < n && g < parts; i++) {
		const uint64_t w = (uint64_t)ents[i].comp_size + ents[i].uncomp_size + 64u;
		while (g < parts && (acc + w) * parts >= total * g) {
			// entry i crosses boundary g: it goes to the side that leaves the smaller imbalance
			const uint64_t target = total * g / parts;
			first[g] = (target - acc) * 2 >= w ? i + 1 : i;
			g++;
		}
		acc += w;
	}
	for (; g <= parts; g++) {
		first[g] = n;
	}
	for (uint32_t k = 1; k <= parts; k++) {   // monotone
		if (first[k] < first[k - 1]) {
			first[k] = first[k - 1];
		}
	}
	return OTZ_SUCCESS;
}

extern "C" int otz_status_accepts(int32_t st, int verify_crc, int ref_compat) {
	if (OTZ_ST_CODE(st) != OTZ_ST_OK) {
		return 0;
	}
	if (ref_compat && (st & OTZ_STF_REF_EOB)) {
		return 0;  // dec:811-816: the reference answers Z_BUF_ERROR
	}
	if (verify_crc && (st & OTZ_STF_CRC_MISMATCH)) {
		return 0;  // otezip.c:670-673
	}
	return 1;
}

// ---------------------------------------------------------------- write path
struct otz_deflate_job {
	bool has_zstd;   // some entry asks for method 93: the compressor instantiation with the Zstandard block writer
	uint32_t n, n_chunks, n_crc_chunks, n_slots;
	uint32_t n_def_chunks;   // chunks [0, n_def_chunks) run on k_deflate_chunks, the best-level chunks behind them on k_deflate_best
	int best_grid;
	uint64_t in_total;
	OtzDflEntry *d_ents;
	OtzDflChunk *d_chunks;
	otz_entry *d_crc_ents;       // the sources described as entries of an "arena" = the input buffer
	OtzCrcChunk *d_crc_chunks;
	OtzEntryState *d_est;
	int32_t *d_status;
	uint32_t *d_acc, *d_crc;
	uint32_t *d_tokens;
	uint8_t *d_cout;
	uint32_t *d_csize;
	uint32_t *d_out_size;
	uint16_t *d_method_out;
	uint64_t *d_out_ofs, *d_total;
	uint8_t *d_dense;
	uint32_t *d_counter;
	int grid;
};

extern "C" void otz_deflate_destroy(otz_ctx *c, otz_deflate_job *j) {
	if (!j) {
		return;
	}
	if (c) {
		cudaSetDevice(c->device);
		cudaStreamSynchronize(c->stream);
	}
	void *ptrs[] = { j->d_ents, j->d_chunks, j->d_crc_ents, j->d_crc_chunks, j->d_est, j->d_status, j->d_acc, j->d_crc, j->d_tokens,
		j->d_cout, j->d_csize, j->d_out_size, j->d_method_out, j->d_out_ofs, j->d_total, j->d_dense, j->d_counter };
	for (void *p : ptrs) {
		cudaFree(p);
	}
	delete j;
}

extern "C" int otz_deflate_plan(otz_ctx *c, const uint64_t *in_ofs, const uint32_t *in_len, const uint16_t *method, uint32_t n,
	otz_deflate_job **out) {
	if (!c || !out || (n && (!in_ofs || !in_len || !method))) {
		return OTZ_ERR_ARG;
	}
	*out = nullptr;
	CK(cudaSetDevice(c->device));
	otz_deflate_job *j = new (std::nothrow) otz_deflate_job();
	if (!j) {
		return OTZ_ERR_NOMEM;
	}
	memset(j, 0, sizeof(*j));
	j->n = n;
	std::vector<OtzDflEntry> ents(n);
	std::vector<OtzDflChunk> chunks;
	std::vector<otz_entry> cents(n);
	std::vector<OtzCrcChunk> cchunks;
	uint64_t total = 0;
	std::vector<OtzDflChunk> bchunks;   // best-level chunks, placed behind all others
	std::vector<uint8_t> is_best(n);
	for (uint32_t i = 0; i < n; i++) {
		const uint16_t m_i = method[i] & (uint16_t)~(OTZ_M_FAST | OTZ_M_BEST);
		const uint32_t fast_i = (method[i] & OTZ_M_FAST) ? 8u : 0u;
		const bool best_i = (method[i] & OTZ_M_BEST) != 0;
		if (m_i != OTZ_M_STORE && m_i != OTZ_M_DEFLATE && m_i != OTZ_M_ZSTD) {
			delete j;
			snprintf(g_err, sizeof(g_err), "otz_deflate_plan: method %u is not on the GPU write path", method[i]);
			return OTZ_ERR_ARG;
		}
		if (best_i && (fast_i || m_i != OTZ_M_DEFLATE)) {
			delete j;
			snprintf(g_err, sizeof(g_err), "otz_deflate_plan: method 0x%x: OTZ_M_BEST is a level of DEFLATE (8) only and excludes OTZ_M_FAST",
				method[i]);
			return OTZ_ERR_ARG;
		}
		std::vector<OtzDflChunk> &cv = best_i ? bchunks : chunks;
		OtzDflEntry &e = ents[i];
		e.in_ofs = in_ofs[i];
		e.len = in_len[i];
		e.method_in = m_i;
		e.pad = 0;
		is_best[i] = best_i;   // (first_chunk counts within bchunks until the two lists are joined)
		e.first_chunk = (uint32_t)cv.size();
		const uint32_t nc = (in_len[i] + DFL_CHUNK - 1) / DFL_CHUNK;
		e.n_chunks = nc;
		for (uint32_t k = 0; k < nc; k++) {
			OtzDflChunk ck;
			ck.in_ofs = in_ofs[i] + (uint64_t)k * DFL_CHUNK;
			ck.len = std::min<uint32_t>(DFL_CHUNK, in_len[i] - k * DFL_CHUNK);
			ck.entry = i;
			ck.last = (k + 1 == nc ? 1u : 0u) | (k == 0 ? 2u : 0u) | (m_i == OTZ_M_ZSTD ? 4u : 0u) | fast_i;
			ck.pad = in_len[i];
			j->has_zstd = j->has_zstd || m_i == OTZ_M_ZSTD;
			cv.push_back(ck);
		}
		otz_entry &ce = cents[i];
		memset(&ce, 0, sizeof(ce));
		ce.out_ofs = in_ofs[i];
		ce.comp_size = ce.uncomp_size = in_len[i];
		ce.method = OTZ_M_DEFLATE;
		const uint32_t ncc = (uint32_t)(((uint64_t)in_len[i] + OTZ_CRC_CHUNK - 1) / OTZ_CRC_CHUNK);
		for (uint32_t k = 0; k < ncc; k++) {
			cchunks.push_back(OtzCrcChunk{ i, k });
		}
		total += in_len[i];
	}
	j->n_def_chunks = (uint32_t)chunks.size();
	for (uint32_t i = 0; i < n; i++) {
		if (is_best[i]) {
			ents[i].first_chunk += j->n_def_chunks;
		}
	}
	chunks.insert(chunks.end(), bchunks.begin(), bchunks.end());
	j->n_chunks = (uint32_t)chunks.size();
	j->n_crc_chunks = (uint32_t)cchunks.size();
	j->in_total = total;
	// persistent grid for the compressor: 2 CTAs x 8 warps per SM
	j->grid = std::max(1, std::min<int>(c->sm_count * 7, (int)((j->n_def_chunks + DFL_WARPS - 1) / DFL_WARPS)));
	j->n_slots = (uint32_t)j->grid * DFL_WARPS;
	// best level: one CTA per chunk, as many as fit the device; the CTAs use token slots of their own, shared with the
	// default kernel, which runs before them on the same stream
	const uint32_t n_best = j->n_chunks - j->n_def_chunks;
	if (n_best) {
		int per_sm = 0;
		CK(cudaFuncSetAttribute(k_deflate_best, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DFB_SMEM));
		CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_deflate_best, DFB_THREADS, DFB_SMEM));
		if (per_sm < 1) {
			otz_deflate_destroy(c, j);
			snprintf(g_err, sizeof(g_err), "otz_deflate_plan: k_deflate_best does not fit an SM");
			return OTZ_ERR_CUDA;
		}
		j->best_grid = (int)std::min<uint32_t>((uint32_t)(c->sm_count * per_sm), n_best);
	}
	const size_t tok_slots = std::max<size_t>(j->n_slots, (size_t)j->best_grid);
	int rc;
	if ((rc = upload(&j->d_ents, ents, c->stream)) || (rc = upload(&j->d_chunks, chunks, c->stream)) ||
		(rc = upload(&j->d_crc_ents, cents, c->stream)) || (rc = upload(&j->d_crc_chunks, cchunks, c->stream))) {
		otz_deflate_destroy(c, j);
		return rc;
	}
	const size_t n1 = std::max<uint32_t>(n, 1), nc1 = std::max<uint32_t>(j->n_chunks, 1);
	bool ok = cudaMalloc(&j->d_est, n1 * sizeof(OtzEntryState)) == cudaSuccess && cudaMalloc(&j->d_status, n1 * 4) == cudaSuccess &&
		cudaMalloc(&j->d_acc, n1 * 4) == cudaSuccess && cudaMalloc(&j->d_crc, n1 * 4) == cudaSuccess &&
		cudaMalloc(&j->d_tokens, tok_slots * DFL_CHUNK * 4) == cudaSuccess &&
		cudaMalloc(&j->d_cout, nc1 * (size_t)DFL_OUT_STRIDE) == cudaSuccess && cudaMalloc(&j->d_csize, nc1 * 4) == cudaSuccess &&
		cudaMalloc(&j->d_out_size, n1 * 4) == cudaSuccess && cudaMalloc(&j->d_method_out, n1 * 2) == cudaSuccess &&
		cudaMalloc(&j->d_out_ofs, n1 * 8) == cudaSuccess && cudaMalloc(&j->d_total, 8) == cudaSuccess &&
		cudaMalloc(&j->d_dense, total + 64) == cudaSuccess && cudaMalloc(&j->d_counter, 64) == cudaSuccess;
	if (!ok) {
		int r = fail_cuda(cudaGetLastError(), "cudaMalloc(deflate job)");
		otz_deflate_destroy(c, j);
		return r;
	}
	CK(cudaMemsetAsync(j->d_status, 0, n1 * 4, c->stream));
	CK(cudaMemsetAsync(j->d_est, 0, n1 * sizeof(OtzEntryState), c->stream));
	CK(cudaStreamSynchronize(c->stream));
	*out = j;
	return OTZ_SUCCESS;
}

extern "C" int otz_deflate_run(otz_ctx *c, otz_deflate_job *j, const uint8_t *d_in, uint64_t in_bytes) {
	if (!c || !j) {
		return OTZ_ERR_ARG;
	}
	(void)in_bytes;
	CK(cudaSetDevice(c->device));
	cudaStream_t s = c->stream;
	const uint32_t n = j->n;
	if (!n) {
		CK(cudaMemsetAsync(j->d_total, 0, 8, s));
		return OTZ_SUCCESS;
	}
	CK(cudaMemsetAsync(j->d_counter, 0, 64, s));
	CK(cudaMemsetAsync(j->d_acc, 0, (size_t)n * 4, s));
	if (j->n_crc_chunks) {
		const uint32_t grid = std::min((uint32_t)c->sm_count * crc_ctas_per_sm(), (j->n_crc_chunks + 7) / 8);
		k_crc_chunks<<<grid, 256, 0, s>>>(nullptr, d_in, j->d_crc_ents, j->d_est, j->d_status, j->d_crc_chunks, j->n_crc_chunks, j->d_acc,
			c->d_tabs, 0, 0);
		c->launches++;
	}
	k_crc_finalize<<<(n + 255) / 256, 256, 0, s>>>(j->d_crc_ents, n, j->d_acc, j->d_crc, j->d_status, c->d_tabs);
	c->launches++;
	if (j->n_def_chunks) {
		const size_t smem = DFL_WARPS * sizeof(DeflateSmem);
		static bool attr_done = false;
		if (!attr_done) {
			CK(cudaFuncSetAttribute(k_deflate_chunks<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
			CK(cudaFuncSetAttribute(k_deflate_chunks<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
			attr_done = true;
		}
		auto kern = j->has_zstd ? k_deflate_chunks<true> : k_deflate_chunks<false>;
		kern<<<j->grid, 32 * DFL_WARPS, smem, s>>>(d_in, j->d_chunks, j->n_def_chunks, j->d_tokens, j->d_cout, j->d_csize, j->d_counter, j->n_slots);
		c->launches++;
	}
	if (j->best_grid) {
		k_deflate_best<<<j->best_grid, DFB_THREADS, DFB_SMEM, s>>>(d_in, j->d_chunks, j->n_def_chunks, j->n_chunks - j->n_def_chunks, j->d_tokens,
			j->d_cout, j->d_csize, j->d_counter + 1);
		c->launches++;
	}
	k_deflate_entry_sizes<<<(n + 255) / 256, 256, 0, s>>>(j->d_ents, n, j->d_csize, j->d_out_size, j->d_method_out);
	k_deflate_scan<<<1, 1024, 0, s>>>(j->d_out_size, n, j->d_out_ofs, j->d_total);
	c->launches += 2;
	if (j->n_chunks) {
		const uint32_t grid = std::min((uint32_t)c->sm_count * 8, (j->n_chunks + 7) / 8);
		k_deflate_gather<<<grid, 256, 0, s>>>(d_in, j->d_cout, j->d_chunks, j->n_chunks, j->d_ents, j->d_csize, j->d_method_out, j->d_out_ofs,
			j->d_dense);
		c->launches++;
	}
	CK(cudaGetLastError());
	return OTZ_SUCCESS;
}

extern "C" int otz_deflate_results(otz_ctx *c, otz_deflate_job *j, uint64_t *out_ofs, uint32_t *out_size, uint32_t *crc, uint16_t *method_out,
	uint64_t *total) {
	if (!c || !j) {
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	cudaStream_t s = c->stream;
	const size_t n = j->n;
	if (n && out_ofs) CK(cudaMemcpyAsync(out_ofs, j->d_out_ofs, n * 8, cudaMemcpyDeviceToHost, s));
	if (n && out_size) CK(cudaMemcpyAsync(out_size, j->d_out_size, n * 4, cudaMemcpyDeviceToHost, s));
	if (n && crc) CK(cudaMemcpyAsync(crc, j->d_crc, n * 4, cudaMemcpyDeviceToHost, s));
	if (n && method_out) CK(cudaMemcpyAsync(method_out, j->d_method_out, n * 2, cudaMemcpyDeviceToHost, s));
	if (total) CK(cudaMemcpyAsync(total, j->d_total, 8, cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	return OTZ_SUCCESS;
}

extern "C" const uint8_t *otz_deflate_device_output(otz_deflate_job *j) { return j ? j->d_dense : nullptr; }

extern "C" int otz_deflate_chunks(otz_ctx *c, otz_deflate_job *j, uint32_t *first_chunk, uint32_t *n_chunks, uint32_t *csize, uint32_t csize_cap,
	uint32_t *chunk_bytes) {
	if (!c || !j) {
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	if (chunk_bytes) {
		*chunk_bytes = DFL_CHUNK;
	}
	if (csize) {
		if (csize_cap < j->n_chunks) {
			return OTZ_ERR_ARG;
		}
		if (j->n_chunks) {
			CK(cudaMemcpyAsync(csize, j->d_csize, (size_t)j->n_chunks * 4, cudaMemcpyDeviceToHost, c->stream));
		}
	}
	if (first_chunk || n_chunks) {
		std::vector<OtzDflEntry> ev(j->n);
		if (j->n) {
			CK(cudaMemcpyAsync(ev.data(), j->d_ents, (size_t)j->n * sizeof(OtzDflEntry), cudaMemcpyDeviceToHost, c->stream));
		}
		CK(cudaStreamSynchronize(c->stream));
		for (uint32_t i = 0; i < j->n; i++) {
			if (first_chunk) {
				first_chunk[i] = ev[i].first_chunk;
			}
			if (n_chunks) {
				n_chunks[i] = ev[i].n_chunks;
			}
		}
	}
	CK(cudaStreamSynchronize(c->stream));
	return (int)j->n_chunks;
}

extern "C" int otz_deflate_fetch(otz_ctx *c, otz_deflate_job *j, uint8_t *out, uint64_t bytes) {
	if (!c || !j || (bytes && !out) || bytes > j->in_total) {
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	if (bytes) {
		CK(cudaMemcpyAsync(out, j->d_dense, bytes, cudaMemcpyDeviceToHost, c->stream));
	}
	CK(cudaStreamSynchronize(c->stream));
	return OTZ_SUCCESS;
}

extern "C" int otz_deflate_host(otz_ctx *c, const uint8_t *in, uint64_t in_bytes, const uint64_t *in_ofs, const uint32_t *in_len,
	const uint16_t *method, uint32_t n, uint8_t *out, uint64_t out_cap, uint64_t *out_ofs, uint32_t *out_size, uint32_t *crc,
	uint16_t *method_out, uint64_t *total) {
	otz_deflate_job *j = nullptr;
	int rc = otz_deflate_plan(c, in_ofs, in_len, method, n, &j);
	if (rc) {
		return rc;
	}
	void *d_in = nullptr;
	uint64_t tot = 0;
	do {
		if ((rc = otz_dev_alloc(c, in_bytes, &d_in))) break;
		if (in_bytes && (rc = otz_h2d(c, d_in, in, in_bytes))) break;
		if ((rc = otz_deflate_run(c, j, (const uint8_t *)d_in, in_bytes))) break;
		if ((rc = otz_deflate_results(c, j, out_ofs, out_size, crc, method_out, &tot))) break;
		if (tot > out_cap) {
			snprintf(g_err, sizeof(g_err), "otz_deflate_host: output needs %llu bytes, capacity %llu", (unsigned long long)tot,
				(unsigned long long)out_cap);
			rc = OTZ_ERR_ARG;
			break;
		}
		rc = otz_deflate_fetch(c, j, out, tot);
	} while (0);
	if (total) {
		*total = tot;
	}
	cudaStreamSynchronize(c->stream);
	if (d_in) {
		cudaFree(d_in);
	}
	otz_deflate_destroy(c, j);
	return rc;
}

// ---------------------------------------------------------------- WinZip AES (k_aes.cuh)
struct OtzAesRun {
	cudaStream_t side;        // the authentication codes run here, beside CTR and the decode
	cudaEvent_t ev[4];        // KDF start, KDF end, CTR end, MAC end
	OtzAesJob *d_jobs;
	OtzAesWork *d_work;
	uint32_t *d_order;
	OtzAesKeys *d_keys;
	int32_t *d_verdict, *d_auth;
	uint8_t *d_pw, *d_salts;
	uint32_t *d_pw_ofs;
	uint64_t pw_bytes;
	uint32_t n;
	bool open_pending;
};

static void aes_free_run(OtzAesRun *r) {
	cudaFree(r->d_jobs);
	cudaFree(r->d_work);
	cudaFree(r->d_order);
	cudaFree(r->d_keys);
	cudaFree(r->d_verdict);
	cudaFree(r->d_auth);
	cudaFree(r->d_pw);
	cudaFree(r->d_salts);
	cudaFree(r->d_pw_ofs);
	r->d_jobs = nullptr;
	r->d_work = nullptr;
	r->d_order = nullptr;
	r->d_keys = nullptr;
	r->d_verdict = r->d_auth = nullptr;
	r->d_pw = r->d_salts = nullptr;
	r->d_pw_ofs = nullptr;
}

static int aes_wipe(otz_ctx *c, OtzAesRun *r);
static void aes_destroy(otz_ctx *c) {
	OtzAesRun *r = c->aes;
	if (!r) {
		return;
	}
	cudaStreamSynchronize(r->side);
	aes_wipe(c, r);
	cudaStreamSynchronize(c->stream);
	aes_free_run(r);
	for (auto &e : r->ev) {
		cudaEventDestroy(e);
	}
	cudaStreamDestroy(r->side);
	delete r;
	c->aes = nullptr;
}

static int aes_run(otz_ctx *c, OtzAesRun **out) {
	if (!c->aes) {
		OtzAesRun *r = new (std::nothrow) OtzAesRun();
		if (!r) {
			return OTZ_ERR_NOMEM;
		}
		c->aes = r;
		CK(cudaStreamCreateWithFlags(&r->side, cudaStreamNonBlocking));
		for (auto &e : r->ev) {
			CK(cudaEventCreate(&e));
		}
	}
	*out = c->aes;
	return OTZ_SUCCESS;
}

static uint32_t aes_salt_bytes(uint16_t strength) { return 4u + 4u * strength; }

// Clear the secrets of a run on the device (round keys, HMAC states, passwords), ordered after its kernels on the stream.
static int aes_wipe(otz_ctx *c, OtzAesRun *r) {
	if (r->n && r->d_keys) {
		CK(cudaMemsetAsync(r->d_keys, 0, sizeof(OtzAesKeys) * r->n, c->stream));
	}
	if (r->pw_bytes && r->d_pw) {
		CK(cudaMemsetAsync(r->d_pw, 0, r->pw_bytes, c->stream));
	}
	return OTZ_SUCCESS;
}

// Upload the jobs, the CTR work list, the longest-first order and the passwords; allocate keys and verdicts.
static int aes_stage(otz_ctx *c, OtzAesRun *r, const std::vector<OtzAesJob> &jobs, const char *const *passwords, uint32_t n_pw) {
	const uint32_t n = (uint32_t)jobs.size();
	std::vector<OtzAesWork> work;
	for (uint32_t i = 0; i < n; i++) {
		const uint32_t nc = std::max<uint32_t>(1, (uint32_t)(((uint64_t)jobs[i].len + OTZ_AES_CHUNK - 1) / OTZ_AES_CHUNK));
		for (uint32_t k = 0; k < nc; k++) {
			work.push_back({ i, k });
		}
	}
	std::vector<uint32_t> order(n);
	for (uint32_t i = 0; i < n; i++) {
		order[i] = i;
	}
	std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return jobs[a].len > jobs[b].len; });
	std::vector<uint32_t> pw_ofs(n_pw + 1, 0);
	std::vector<uint8_t> pw;
	for (uint32_t k = 0; k < n_pw; k++) {
		const char *p = passwords[k] ? passwords[k] : "";
		pw.insert(pw.end(), p, p + strlen(p));
		pw_ofs[k + 1] = (uint32_t)pw.size();
	}
	r->n = n;
	r->pw_bytes = pw.size();
	int rc;
	if ((rc = upload(&r->d_jobs, jobs, c->stream)) != OTZ_SUCCESS || (rc = upload(&r->d_work, work, c->stream)) != OTZ_SUCCESS ||
		(rc = upload(&r->d_order, order, c->stream)) != OTZ_SUCCESS || (rc = upload(&r->d_pw, pw, c->stream)) != OTZ_SUCCESS ||
		(rc = upload(&r->d_pw_ofs, pw_ofs, c->stream)) != OTZ_SUCCESS) {
		return rc;
	}
	std::fill(pw.begin(), pw.end(), 0);   // (the host copy of the passwords)
	CK(cudaMalloc(&r->d_keys, sizeof(OtzAesKeys) * std::max<uint32_t>(n, 1)));
	CK(cudaMalloc(&r->d_verdict, sizeof(int32_t) * std::max<uint32_t>(n, 1)));
	CK(cudaMalloc(&r->d_auth, sizeof(int32_t) * std::max<uint32_t>(n, 1)));
	CK(cudaMemsetAsync(r->d_auth, 0, sizeof(int32_t) * std::max<uint32_t>(n, 1), c->stream));
	return OTZ_SUCCESS;
}

extern "C" int otz_aes_open(otz_ctx *c, const uint8_t *d_src, uint64_t src_len, const otz_aes_entry *ents, uint32_t n,
	const char *const *passwords, uint32_t n_pw, uint8_t *d_plain, uint64_t plain_len) {
	if (!c || (n && (!ents || !d_src || !d_plain)) || (n_pw && !passwords) || n_pw >= OTZ_AES_NOPASSWORD) {
		snprintf(g_err, sizeof(g_err), "otz_aes_open: missing buffer or more than %u passwords", OTZ_AES_NOPASSWORD - 1);
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	OtzAesRun *r;
	int rc = aes_run(c, &r);
	if (rc != OTZ_SUCCESS) {
		return rc;
	}
	if (r->open_pending) {
		snprintf(g_err, sizeof(g_err), "otz_aes_open: the previous run was not collected with otz_aes_status");
		return OTZ_ERR_ARG;
	}
	CK(cudaStreamSynchronize(r->side));
	aes_free_run(r);
	std::vector<OtzAesJob> jobs(n);
	for (uint32_t i = 0; i < n; i++) {
		const otz_aes_entry &e = ents[i];
		const uint32_t sl = aes_salt_bytes(e.strength);
		if (e.strength < 1 || e.strength > 3 || e.size < sl + 2 + 10 || e.payload_ofs > src_len || src_len - e.payload_ofs < e.size ||
			e.data_ofs > plain_len || plain_len - e.data_ofs < 30ull + e.size - sl - 12) {
			snprintf(g_err, sizeof(g_err), "otz_aes_open: entry %u outside its buffers or of unknown strength", i);
			return OTZ_ERR_ARG;
		}
		OtzAesJob &j = jobs[i];
		j.salt = e.payload_ofs;
		j.pwv = e.payload_ofs + sl;
		j.src = e.payload_ofs + sl + 2;
		j.len = e.size - sl - 12;
		j.mac = j.src + j.len;
		j.hdr = e.data_ofs;
		j.dst = e.data_ofs + 30;
		j.strength = e.strength;
		j.pw = e.password < n_pw ? e.password : (uint16_t)OTZ_AES_NOPW;
	}
	if ((rc = aes_stage(c, r, jobs, passwords, n_pw)) != OTZ_SUCCESS) {
		return rc;
	}
	CK(cudaEventRecord(r->ev[0], c->stream));
	if (n) {
		k_aes_kdf<<<(4 * n + OTZ_AES_KDF_THREADS - 1) / OTZ_AES_KDF_THREADS, OTZ_AES_KDF_THREADS, 0, c->stream>>>(r->d_jobs, n, r->d_pw,
			r->d_pw_ofs, n_pw, d_src, const_cast<uint8_t *>(d_src), src_len, 0, r->d_keys, r->d_verdict);
		CK(cudaGetLastError());
		c->launches++;
	}
	CK(cudaEventRecord(r->ev[1], c->stream));
	CK(cudaStreamWaitEvent(r->side, r->ev[1], 0));
	if (n) {
		uint32_t nw = 0;
		for (const OtzAesJob &j : jobs) {
			nw += std::max<uint32_t>(1, (uint32_t)(((uint64_t)j.len + OTZ_AES_CHUNK - 1) / OTZ_AES_CHUNK));
		}
		k_aes_ctr<<<nw, OTZ_AES_CTR_THREADS, 0, c->stream>>>(r->d_jobs, n, r->d_work, nw, r->d_keys, r->d_verdict, d_src, src_len,
			d_plain, plain_len, 1);
		CK(cudaGetLastError());
		k_aes_mac<<<(n + 127) / 128, 128, 0, r->side>>>(r->d_jobs, r->d_order, n, r->d_keys, r->d_verdict, d_src,
			const_cast<uint8_t *>(d_src), src_len, 0, r->d_auth);
		CK(cudaGetLastError());
		c->launches += 2;
	}
	CK(cudaEventRecord(r->ev[2], c->stream));
	CK(cudaEventRecord(r->ev[3], r->side));
	r->open_pending = true;
	return OTZ_SUCCESS;
}

extern "C" int otz_aes_status(otz_ctx *c, int32_t *status) {
	if (!c || !c->aes || !c->aes->open_pending) {
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	OtzAesRun *r = c->aes;
	r->open_pending = false;
	CK(cudaStreamWaitEvent(c->stream, r->ev[3], 0));
	const uint32_t n = r->n;
	std::vector<int32_t> v(std::max<uint32_t>(n, 1)), a(std::max<uint32_t>(n, 1));
	int rc = aes_wipe(c, r);
	if (rc != OTZ_SUCCESS) {
		return rc;
	}
	if (n) {
		CK(cudaMemcpyAsync(v.data(), r->d_verdict, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, c->stream));
		CK(cudaMemcpyAsync(a.data(), r->d_auth, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, c->stream));
	}
	CK(cudaStreamSynchronize(c->stream));
	for (uint32_t i = 0; status && i < n; i++) {
		status[i] = v[i] != OTZ_ST_OK ? v[i] : a[i] ? OTZ_ST_AUTH : OTZ_ST_OK;
	}
	return OTZ_SUCCESS;
}

extern "C" int otz_aes_times(otz_ctx *c, float *ms_kdf, float *ms_ctr, float *ms_mac) {
	if (!c || !c->aes) {
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	OtzAesRun *r = c->aes;
	CK(cudaEventSynchronize(r->ev[3]));
	CK(cudaEventSynchronize(r->ev[2]));
	if (ms_kdf) {
		CK(cudaEventElapsedTime(ms_kdf, r->ev[0], r->ev[1]));
	}
	if (ms_ctr) {
		CK(cudaEventElapsedTime(ms_ctr, r->ev[1], r->ev[2]));
	}
	if (ms_mac) {
		CK(cudaEventElapsedTime(ms_mac, r->ev[1], r->ev[3]));
	}
	return OTZ_SUCCESS;
}

extern "C" int otz_aes_seal(otz_ctx *c, const uint8_t *d_in, uint64_t in_len, const otz_aes_entry *ents, uint32_t n, const uint8_t *salts,
	const char *const *passwords, uint32_t n_pw, uint8_t *d_out, uint64_t out_len) {
	if (!c || (n && (!ents || !salts || !d_out)) || (n_pw && !passwords) || n_pw >= OTZ_AES_NOPASSWORD) {
		snprintf(g_err, sizeof(g_err), "otz_aes_seal: missing buffer or more than %u passwords", OTZ_AES_NOPASSWORD - 1);
		return OTZ_ERR_ARG;
	}
	CK(cudaSetDevice(c->device));
	OtzAesRun *r;
	int rc = aes_run(c, &r);
	if (rc != OTZ_SUCCESS) {
		return rc;
	}
	if (r->open_pending) {
		snprintf(g_err, sizeof(g_err), "otz_aes_seal: the previous otz_aes_open was not collected with otz_aes_status");
		return OTZ_ERR_ARG;
	}
	CK(cudaStreamSynchronize(r->side));
	aes_free_run(r);
	std::vector<OtzAesJob> jobs(n);
	for (uint32_t i = 0; i < n; i++) {
		const otz_aes_entry &e = ents[i];
		const uint32_t sl = aes_salt_bytes(e.strength);
		if (e.strength < 1 || e.strength > 3 || e.password >= n_pw || (e.size && !d_in) || e.data_ofs > in_len || in_len - e.data_ofs < e.size ||
			e.payload_ofs > out_len || out_len - e.payload_ofs < (uint64_t)e.size + sl + 12) {
			snprintf(g_err, sizeof(g_err), "otz_aes_seal: entry %u outside its buffers, of unknown strength or without a password", i);
			return OTZ_ERR_ARG;
		}
		OtzAesJob &j = jobs[i];
		j.salt = 16ull * i;
		j.hdr = e.payload_ofs;
		j.pwv = e.payload_ofs + sl;
		j.dst = e.payload_ofs + sl + 2;
		j.src = e.data_ofs;
		j.len = e.size;
		j.mac = j.dst + j.len;
		j.strength = e.strength;
		j.pw = e.password;
	}
	if ((rc = aes_stage(c, r, jobs, passwords, n_pw)) != OTZ_SUCCESS) {
		return rc;
	}
	if (n) {
		std::vector<uint8_t> sv(salts, salts + 16ull * n);
		if ((rc = upload(&r->d_salts, sv, c->stream)) != OTZ_SUCCESS) {
			return rc;
		}
		uint32_t nw = 0;
		for (const OtzAesJob &j : jobs) {
			nw += std::max<uint32_t>(1, (uint32_t)(((uint64_t)j.len + OTZ_AES_CHUNK - 1) / OTZ_AES_CHUNK));
		}
		k_aes_kdf<<<(4 * n + OTZ_AES_KDF_THREADS - 1) / OTZ_AES_KDF_THREADS, OTZ_AES_KDF_THREADS, 0, c->stream>>>(r->d_jobs, n, r->d_pw,
			r->d_pw_ofs, n_pw, r->d_salts, d_out, out_len, 1, r->d_keys, r->d_verdict);
		CK(cudaGetLastError());
		k_aes_ctr<<<nw, OTZ_AES_CTR_THREADS, 0, c->stream>>>(r->d_jobs, n, r->d_work, nw, r->d_keys, r->d_verdict, d_in, in_len, d_out,
			out_len, 0);
		CK(cudaGetLastError());
		k_aes_mac<<<(n + 127) / 128, 128, 0, c->stream>>>(r->d_jobs, r->d_order, n, r->d_keys, r->d_verdict, d_out, d_out, out_len, 1, r->d_auth);
		CK(cudaGetLastError());
		c->launches += 3;
	}
	if ((rc = aes_wipe(c, r)) != OTZ_SUCCESS) {
		return rc;
	}
	CK(cudaStreamSynchronize(c->stream));
	return OTZ_SUCCESS;
}

/*
 * crgpu_api.cu — C ABI of libcrgpu.so (include/crgpu.h): scene upload, the per-tile wavefront driver,
 * framebuffer access.  Host code here only lays data out in HBM and launches kernels; all arithmetic
 * of the hot path is in the kernels (crgpu_kernels.cuh).  No CPU fallback exists.
 */
#include "../../include/crgpu.h"
#include "crgpu_wave.cuh"
#include "crgpu_scene.cuh"

#define CRG_HITKAT_BYTES 160
#define CRG_TAIL_FROM 6      /* first bounce at which the tail kernel may take over (it only does when <= 16384 rays are left) */

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cstdarg>
#include <vector>
#include <queue>
#include <thread>
#include <mutex>

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
	va_list vl;
	va_start(vl, fmt);
	vsnprintf(g_err, sizeof g_err, fmt, vl);
	va_end(vl);
	return code;
}
/* the same for the other translation units of libcrgpu.so (crgpu_bvh_build.cu) */
int crg_fail(int code, const char *fmt, ...) {
	va_list vl;
	va_start(vl, fmt);
	vsnprintf(g_err, sizeof g_err, fmt, vl);
	va_end(vl);
	return code;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(CRGPU_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)

extern "C" const char *crgpu_last_error(void) { return g_err; }

extern "C" int crgpu_device_count(int *n) {
	if (!n) return fail(CRGPU_ERR_BAD_ARGUMENT, "n is NULL");
	int c = 0;
	cudaError_t e = cudaGetDeviceCount(&c);
	if (e != cudaSuccess || c < 1) { *n = 0; return fail(CRGPU_ERR_NO_DEVICE, "no CUDA device: %s", cudaGetErrorString(e)); }
	*n = c;
	return CRGPU_OK;
}

/* ---- per-device context: a caching allocator ----------------------------------------------------------------------------------
 * A frame of this renderer wants ~35 GB of wavefront state, a 50 MB scene and a framebuffer.  cudaMalloc of those costs
 * 10-55 ms and cudaFree of the 35 GB 0.3-0.5 s (profiles/r01_e2e_breakdown.txt) — per FRAME when every renderFrame creates and
 * destroys its scene replica, as the reference's renderFrame does with its buffers.  So device memory released by a scene goes
 * back to a per-device cache and the next scene on that device takes it from there (best fit within 2x); a cudaMalloc that
 * fails trims the cache and retries.  crgpu_device_trim() hands everything back to the driver. */
#define CRG_MAX_DEVICES 64
struct DevBlock { void *p; size_t bytes; };
struct DevCtx {
	std::mutex lock;
	std::vector<DevBlock> cache;
	size_t cached = 0;
};
static DevCtx g_ctx[CRG_MAX_DEVICES];
static DevCtx &ctx_of(int dev) { return g_ctx[dev >= 0 && dev < CRG_MAX_DEVICES ? dev : 0]; }

static void ctx_trim_locked(DevCtx &c) {
	for (DevBlock &b : c.cache) cudaFree(b.p);
	c.cache.clear();
	c.cached = 0;
}
/* the calling thread's current device must be `dev` */
static int ctx_alloc(int dev, size_t bytes, void **out) {
	*out = nullptr;
	if (bytes == 0) bytes = 256;
	DevCtx &c = ctx_of(dev);
	std::lock_guard<std::mutex> g(c.lock);
	int best = -1;
	for (size_t i = 0; i < c.cache.size(); ++i)
		if (c.cache[i].bytes >= bytes && c.cache[i].bytes <= 2 * bytes + (1u << 20) && (best < 0 || c.cache[i].bytes < c.cache[(size_t)best].bytes)) best = (int)i;
	if (best >= 0) {
		*out = c.cache[(size_t)best].p;
		c.cached -= c.cache[(size_t)best].bytes;
		c.cache.erase(c.cache.begin() + best);
		return CRGPU_OK;
	}
	cudaError_t e = cudaMalloc(out, bytes);
	if (e == cudaErrorMemoryAllocation && !c.cache.empty()) {
		cudaGetLastError();
		ctx_trim_locked(c);
		e = cudaMalloc(out, bytes);
	}
	if (e == cudaErrorMemoryAllocation) { cudaGetLastError(); *out = nullptr; return fail(CRGPU_ERR_NOMEM, "out of device memory allocating %zu bytes on device %d", bytes, dev); }
	if (e != cudaSuccess) { *out = nullptr; return fail(CRGPU_ERR_CUDA, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e)); }
	return CRGPU_OK;
}
/* size actually backing a pointer handed out for a request of `bytes` is not tracked: callers remember their request, and a
 * cached block is re-used only for requests it can hold, so recording the REQUEST size is conservative and safe */
static void ctx_free(int dev, void *p, size_t bytes) {
	if (!p) return;
	if (bytes == 0) bytes = 256;
	DevCtx &c = ctx_of(dev);
	std::lock_guard<std::mutex> g(c.lock);
	if (c.cache.size() >= 24) {                      /* bound the list: drop the smallest entry */
		size_t k = 0;
		for (size_t i = 1; i < c.cache.size(); ++i) if (c.cache[i].bytes < c.cache[k].bytes) k = i;
		cudaFree(c.cache[k].p);
		c.cached -= c.cache[k].bytes;
		c.cache.erase(c.cache.begin() + (long)k);
	}
	c.cache.push_back({ p, bytes });
	c.cached += bytes;
}
static size_t ctx_cached_bytes(int dev) { DevCtx &c = ctx_of(dev); std::lock_guard<std::mutex> g(c.lock); return c.cached; }

extern "C" int crgpu_device_trim(int device) {
	int ndev = 0;
	int rc = crgpu_device_count(&ndev);
	if (rc) return rc;
	if (device < 0 || device >= ndev) return fail(CRGPU_ERR_BAD_ARGUMENT, "device %d out of range (have %d)", device, ndev);
	CU(cudaSetDevice(device));
	DevCtx &c = ctx_of(device);
	std::lock_guard<std::mutex> g(c.lock);
	ctx_trim_locked(c);
	return CRGPU_OK;
}

/* pinned host memory for buffers that cross PCIe every frame (the host framebuffer of renderFrame, the prepared scene) */
extern "C" void *crgpu_host_alloc(size_t bytes) {
	void *p = nullptr;
	if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
	return p;
}
extern "C" void crgpu_host_free(void *p) { if (p) cudaFreeHost(p); }

/* ---- the prepared scene: the flat scene re-laid out for the kernels, in ONE host slab (pinned) ----------------------------------
 * crgpu_prepare() does everything about a scene that does not depend on the device: validation, BVH re-layout into pair nodes,
 * triangle packing, shading records.  crgpu_scene_create_prepared() is then one host->device copy of the slab plus two small
 * pointer-carrying tables.  A host that renders many frames of one scene, or one frame on many GPUs, prepares once. */
enum { SEC_PAIRS, SEC_TRIS, SEC_SLOT_POLY, SEC_SPOLYS, SEC_TOP_PRIMS, SEC_BVHS, SEC_INSTS, SEC_MATS, SEC_NODES, SEC_TEXS, SEC_LUT, SEC_TEXDATA, SEC_COUNT };
struct crgpu_prepared {
	crs_prefs prefs;
	crs_camera camera;
	int32_t background;
	uint32_t instance_count;
	DevBvh top;
	uint32_t texture_count;
	bool xnodes;               /* some node is of a kind only the complete interpreter (NodeX) evaluates */
	uint8_t *slab;
	bool pinned;
	size_t slab_bytes;
	size_t off[SEC_COUNT], len[SEC_COUNT];
};

struct crgpu_scene {
	int device;
	int sm_count;
	bool xnodes;               /* crgpu_prepared::xnodes: selects the K3 / tail kernels with the complete node interpreter */
	cudaStream_t stream;       /* the stream work is enqueued on (own_stream unless crgpu_set_stream) */
	cudaStream_t own_stream;
	unsigned long long fetched[8];   /* device counters at the previous stats fetch */
	uint64_t pend_paths, pend_launches;
	float pend_trace_ms, pend_shade_ms, pend_total_ms;
	DevScene dev;
	DevScene *dev_copy;        /* the same descriptor in HBM, for kernels that call noinline device functions */
	void *slab; size_t slab_bytes;   /* the scene arrays + dev_copy */
	void *small; size_t small_bytes; /* hist, counts, stats */
	float *fb;                 /* W*H*3 fp32, row H-1-y */
	uint8_t *fb8;              /* lazily allocated sRGB8 staging */
	size_t fb_floats;
	uint64_t max_paths;
	uint64_t cap_paths;        /* capacity of the wavefront buffers */
	void *wave; size_t wave_bytes;
	int wave_sets;             /* 1, or 2 when batches are overlapped on two streams (each set holds cap_paths paths) */
	WaveBuffers wb;            /* set 0 */
	WaveBuffers wb2;           /* set 1: own ray / hit / radiance buffers and own hist + counts; stats shared */
	cudaStream_t stream2;      /* the second stream of overlapped batches */
	cudaEvent_t ev[4];
	cudaEvent_t evAcc[2], evFork;   /* accumulate-order chain between the two streams */
	uint32_t *pixels;          /* device pixel list of the last crgpu_render_tiles tile set */
	size_t pixel_cap;
	std::vector<int> pixel_key;
};

/* ---- node graph checks -------------------------------------------------------------------------------------- */
static bool node_ok(const crs_scene *f, int idx) { return idx >= 0 && (uint32_t)idx < f->node_count; }

/* Nesting as the device counts it (crgpu_shade.cuh).  The hot interpreter NodeEval<CRG_NODE_DEPTH> knows the node kinds of JSON
 * scenes: color->value->color recursion costs a level at checker/blackbody -> value (grayscale/alpha -> color and the checker's
 * A/B tail calls are free).  At the first node of any other kind the complete interpreter NodeX<CRG_XNODE_DEPTH> takes over, where
 * EVERY edge costs a level (xnode_depth) whatever the kinds below. */
static int xnode_depth(const crs_scene *f, int idx, int guard) {
	if (!node_ok(f, idx) || guard > 64) return 1000;
	const crs_node &n = f->nodes[idx];
	int ins = 0;
	switch (n.kind) {
	case CRS_COLOR_CONSTANT: case CRS_COLOR_IMAGE: case CRS_COLOR_GRADIENT: case CRS_VALUE_CONSTANT: case CRS_VALUE_RAYLENGTH:
	case CRS_VECTOR_CONSTANT: case CRS_VECTOR_NORMAL: return 0;
	case CRS_COLOR_CHECKER: case CRS_COLOR_COMBINE_RGB: ins = 3; break;
	case CRS_VALUE_MATH: if (n.options >= CRS_MATH_OP_COUNT) return 1000; ins = 2; break;
	case CRS_VECTOR_VECMATH: if (n.options >= CRS_VEC_OP_COUNT) return 1000; ins = 2; break;
	case CRS_COLOR_BLACKBODY: case CRS_COLOR_COMBINE_VALUE: case CRS_COLOR_VECTOCOLOR: case CRS_VALUE_GRAYSCALE: case CRS_VALUE_ALPHA: ins = 1; break;
	case CRS_VALUE_FRESNEL: {                            /* in1 (normal) is never evaluated (fresnel.c:43-55) but must be a vector node */
		if (!node_ok(f, n.in[1])) return 1000;
		const int k = f->nodes[n.in[1]].kind;
		if (k != CRS_VECTOR_CONSTANT && k != CRS_VECTOR_NORMAL && k != CRS_VECTOR_VECMATH) return 1000;
		ins = 1; break;
	}
	default: return 1000;
	}
	/* operand classes: what each input must be */
	int m = 0;
	for (int k = 0; k < ins; ++k) {
		if (!node_ok(f, n.in[k])) return 1000;
		const int ck = f->nodes[n.in[k]].kind;
		const bool is_color = ck >= CRS_COLOR_CONSTANT && ck <= CRS_COLOR_COMBINE_RGB, is_value = ck >= CRS_VALUE_CONSTANT && ck <= CRS_VALUE_RAYLENGTH,
				   is_vector = ck >= CRS_VECTOR_CONSTANT && ck <= CRS_VECTOR_VECMATH;
		bool ok;
		switch (n.kind) {
		case CRS_COLOR_CHECKER: ok = k < 2 ? is_color : is_value; break;
		case CRS_VALUE_GRAYSCALE: case CRS_VALUE_ALPHA: ok = is_color; break;
		case CRS_COLOR_VECTOCOLOR: case CRS_VECTOR_VECMATH: ok = is_vector; break;
		default: ok = is_value; break;                   /* blackbody, combine, combine rgb, math, fresnel (IOR) */
		}
		if (!ok) return 1000;
		const int d = xnode_depth(f, n.in[k], guard + 1);
		if (d > m) m = d;
	}
	return 1 + m;
}
static int xnode_entry(const crs_scene *f, int idx, int guard) { return xnode_depth(f, idx, guard) <= CRG_XNODE_DEPTH ? 0 : 1000; }
static int value_depth(const crs_scene *f, int idx, int guard);
static int color_depth(const crs_scene *f, int idx, int guard) {
	if (!node_ok(f, idx) || guard > 64) return 1000;
	const crs_node &n = f->nodes[idx];
	switch (n.kind) {
	case CRS_COLOR_CONSTANT: case CRS_COLOR_IMAGE: case CRS_COLOR_GRADIENT: return 0;
	case CRS_COLOR_CHECKER: {
		int a = color_depth(f, n.in[0], guard + 1), b = color_depth(f, n.in[1], guard + 1);
		int v = 1 + value_depth(f, n.in[2], guard + 1);
		int m = a > b ? a : b;
		return m > v ? m : v;
	}
	case CRS_COLOR_BLACKBODY: return 1 + value_depth(f, n.in[0], guard + 1);
	case CRS_COLOR_VECTOCOLOR: case CRS_COLOR_COMBINE_VALUE: case CRS_COLOR_COMBINE_RGB: return xnode_entry(f, idx, guard);
	default: return 1000;
	}
}
static int value_depth(const crs_scene *f, int idx, int guard) {
	if (!node_ok(f, idx) || guard > 64) return 1000;
	const crs_node &n = f->nodes[idx];
	switch (n.kind) {
	case CRS_VALUE_CONSTANT: return 0;
	case CRS_VALUE_GRAYSCALE: case CRS_VALUE_ALPHA: return color_depth(f, n.in[0], guard + 1);
	case CRS_VALUE_MATH: case CRS_VALUE_FRESNEL: case CRS_VALUE_RAYLENGTH: return xnode_entry(f, idx, guard);
	default: return 1000;
	}
}
static bool color_reads_uv(const crs_scene *f, int idx);
static bool value_reads_uv(const crs_scene *f, int idx) {
	if (!node_ok(f, idx)) return false;
	const crs_node &n = f->nodes[idx];
	switch (n.kind) {
	case CRS_VALUE_GRAYSCALE: case CRS_VALUE_ALPHA: return color_reads_uv(f, n.in[0]);
	case CRS_VALUE_MATH: return value_reads_uv(f, n.in[0]) || value_reads_uv(f, n.in[1]);
	case CRS_VALUE_FRESNEL: return value_reads_uv(f, n.in[0]);
	default: return false;
	}
}
static bool color_reads_uv(const crs_scene *f, int idx) {
	if (!node_ok(f, idx)) return false;
	const crs_node &n = f->nodes[idx];
	switch (n.kind) {
	case CRS_COLOR_IMAGE: case CRS_COLOR_CHECKER: return true;
	case CRS_COLOR_BLACKBODY: case CRS_COLOR_COMBINE_VALUE: return value_reads_uv(f, n.in[0]);
	case CRS_COLOR_COMBINE_RGB: return value_reads_uv(f, n.in[0]) || value_reads_uv(f, n.in[1]) || value_reads_uv(f, n.in[2]);
	default: return false;            /* vector nodes never read uv */
	}
}
/* validates a bsdf tree; *add_depth = nesting of ADD nodes; *uv = some node reads uv */
static int check_bsdf(const crs_scene *f, int idx, int add_level, int guard, bool *uv) {
	if (!node_ok(f, idx) || guard > 64) return fail(CRGPU_ERR_UNSUPPORTED, "bsdf node index %d out of range or graph too deep", idx);
	const crs_node &n = f->nodes[idx];
	auto col = [&](int c) -> int {
		if (color_depth(f, c, 0) > CRG_NODE_DEPTH) return fail(CRGPU_ERR_UNSUPPORTED, "color node %d nests deeper than %d", c, CRG_NODE_DEPTH);
		if (color_reads_uv(f, c)) *uv = true;
		return 0;
	};
	auto val = [&](int v) -> int {
		if (value_depth(f, v, 0) > CRG_NODE_DEPTH) return fail(CRGPU_ERR_UNSUPPORTED, "value node %d nests deeper than %d", v, CRG_NODE_DEPTH);
		if (value_reads_uv(f, v)) *uv = true;
		return 0;
	};
	int rc;
	switch (n.kind) {
	case CRS_BSDF_DIFFUSE: case CRS_BSDF_TRANSPARENT: case CRS_BSDF_ISOTROPIC: return col(n.in[0]);
	case CRS_BSDF_METAL: case CRS_BSDF_EMISSIVE: if ((rc = col(n.in[0]))) return rc; return val(n.in[1]);
	case CRS_BSDF_GLASS: case CRS_BSDF_BACKGROUND:
		if ((rc = col(n.in[0]))) return rc; if ((rc = val(n.in[1]))) return rc; return val(n.in[2]);
	case CRS_BSDF_PLASTIC:
		if ((rc = col(n.in[0]))) return rc; if ((rc = col(n.in[1]))) return rc;
		return check_bsdf(f, n.in[2], add_level, guard + 1, uv);
	case CRS_BSDF_MIX:
		if ((rc = val(n.in[2]))) return rc;
		if ((rc = check_bsdf(f, n.in[0], add_level, guard + 1, uv))) return rc;
		return check_bsdf(f, n.in[1], add_level, guard + 1, uv);
	case CRS_BSDF_ADD:
		if (2 * (add_level + 1) > CRG_ADD_STACK) return fail(CRGPU_ERR_UNSUPPORTED, "ADD nodes nest deeper than %d", CRG_ADD_STACK / 2);
		if ((rc = check_bsdf(f, n.in[0], add_level + 1, guard + 1, uv))) return rc;
		return check_bsdf(f, n.in[1], add_level + 1, guard + 1, uv);
	default: return fail(CRGPU_ERR_UNSUPPORTED, "node %d has kind %d where a bsdf is expected", idx, n.kind);
	}
}

/* ---- BVH re-layout: reference nodes (bvh.c:37-42) -> BFS-ordered PairNodes ---------------------------------------- */
/* errors raised on worker threads (fail() writes a thread-local buffer): first one wins, reported by the caller */
struct HostError {
	std::mutex lock;
	int code = 0;
	char msg[256] = "";
	int set(int c, const char *m) { std::lock_guard<std::mutex> g(lock); if (!code) { code = c; snprintf(msg, sizeof msg, "%s", m); } return c; }
};

/* fn(lo, hi) over [0, n) on a few host threads (CRGPU_HOST_THREADS, default min(hardware, 16)); small n stays inline */
template <class F>
static void host_parallel_for(uint32_t n, F fn) {
	static const unsigned want = [] {
		const char *e = getenv("CRGPU_HOST_THREADS");
		unsigned t = e ? (unsigned)atoi(e) : std::thread::hardware_concurrency();
		return t < 1u ? 1u : (t > 16u ? 16u : t);
	}();
	const unsigned threads = n < 16384u ? 1u : want;
	if (threads <= 1u) { fn(0u, n); return; }
	std::vector<std::thread> pool;
	for (unsigned k = 1; k < threads; ++k)
		pool.emplace_back(fn, (uint32_t)((uint64_t)n * k / threads), (uint32_t)((uint64_t)n * (k + 1) / threads));
	fn(0u, (uint32_t)((uint64_t)n / threads));
	for (auto &t : pool) t.join();
}

static int build_pairs(const crs_scene *f, const crs_bvh &b, std::vector<PairNode> &pairs, DevBvh &out, uint32_t slot_offset, HostError *err) {
	memset(&out, 0, sizeof out);
	out.pair_offset = (uint32_t)pairs.size();
	out.pair_end = out.pair_offset;
	out.node_count = b.node_count;
	out.slot_offset = slot_offset;
	if (b.node_count == 0) return CRGPU_OK;
	const crs_bvh_node *nodes = f->bvh_nodes + b.node_offset;
	if (b.node_count == 1) {
		memcpy(out.root_bounds, nodes[0].bounds, sizeof out.root_bounds);
		out.root_first = nodes[0].first_child_or_prim;
		out.root_count = nodes[0].prim_count_leaf & CRS_BVH_COUNT_MASK;
		if ((uint64_t)out.root_first + out.root_count > (uint64_t)b.prim_count) return err->set(CRGPU_ERR_BAD_ARGUMENT, "BVH leaf range outside the primitive list");
		return CRGPU_OK;
	}
	/* BFS over internal nodes; pair index = BFS rank */
	std::vector<uint32_t> order;            /* reference node index of each internal node, BFS order */
	order.reserve(b.node_count / 2 + 1);
	std::vector<uint32_t> rank(b.node_count, 0xffffffffu);
	std::vector<uint8_t> depth(b.node_count, 0);   /* the traversal stack holds CRG_MAX_STACK entries per level (bvh.c:32) */
	order.push_back(0);
	rank[0] = 0;
	for (size_t head = 0; head < order.size(); ++head) {
		const crs_bvh_node &n = nodes[order[head]];
		if (n.prim_count_leaf & CRS_BVH_LEAF_BIT) return err->set(CRGPU_ERR_BAD_ARGUMENT, "BVH root/internal node is a leaf");
		const uint32_t fc = n.first_child_or_prim;
		if ((uint64_t)fc + 1u >= (uint64_t)b.node_count) return err->set(CRGPU_ERR_BAD_ARGUMENT, "BVH child index out of range");
		if (depth[order[head]] >= CRG_MAX_STACK) return err->set(CRGPU_ERR_UNSUPPORTED, "BVH deeper than 64 levels");
		for (uint32_t k = 0; k < 2; ++k) {
			const crs_bvh_node &c = nodes[fc + k];
			if (!(c.prim_count_leaf & CRS_BVH_LEAF_BIT)) {
				if (rank[fc + k] != 0xffffffffu) return err->set(CRGPU_ERR_BAD_ARGUMENT, "BVH is not a tree");
				rank[fc + k] = (uint32_t)order.size();
				depth[fc + k] = (uint8_t)(depth[order[head]] + 1);
				order.push_back(fc + k);
			} else if ((uint64_t)c.first_child_or_prim + (uint64_t)(c.prim_count_leaf & CRS_BVH_COUNT_MASK) > (uint64_t)b.prim_count) {
				return err->set(CRGPU_ERR_BAD_ARGUMENT, "BVH leaf range outside the primitive list");
			}
		}
	}
	const size_t first = pairs.size();
	pairs.resize(first + order.size());
	host_parallel_for((uint32_t)order.size(), [&](uint32_t lo, uint32_t hi) {
		for (uint32_t r = lo; r < hi; ++r) {
			const crs_bvh_node &n = nodes[order[r]];
			const uint32_t fc = n.first_child_or_prim;
			PairNode p;
			memset(&p, 0, sizeof p);
			const crs_bvh_node &l = nodes[fc], &rr = nodes[fc + 1];
			memcpy(p.lb, l.bounds, sizeof p.lb);
			memcpy(p.rb, rr.bounds, sizeof p.rb);
			if (l.prim_count_leaf & CRS_BVH_LEAF_BIT) { p.lref = l.first_child_or_prim; p.lmeta = CRG_LEAF_BIT | (l.prim_count_leaf & CRS_BVH_COUNT_MASK); }
			else { p.lref = rank[fc]; p.lmeta = 0; }
			if (rr.prim_count_leaf & CRS_BVH_LEAF_BIT) { p.rref = rr.first_child_or_prim; p.rmeta = CRG_LEAF_BIT | (rr.prim_count_leaf & CRS_BVH_COUNT_MASK); }
			else { p.rref = rank[fc + 1]; p.rmeta = 0; }
			pairs[first + r] = p;
		}
	});
	out.pair_end = (uint32_t)pairs.size();
	return CRGPU_OK;
}

static inline void f3(float *dst, const float *src, size_t idx) { dst[0] = src[3 * idx]; dst[1] = src[3 * idx + 1]; dst[2] = src[3 * idx + 2]; }

/* all wavefront buffers of a scene are carved from ONE device block (one cudaMalloc / one cache hit per frame) */
static int alloc_wave(crgpu_scene *s, uint64_t paths, int sets) {
	if (paths <= s->cap_paths && sets <= s->wave_sets) return CRGPU_OK;
	if (s->wave) {
		cudaStreamSynchronize(s->stream);                           /* queued kernels may still use the old block */
		if (s->stream2) cudaStreamSynchronize(s->stream2);
		ctx_free(s->device, s->wave, s->wave_bytes);
	}
	s->wave = nullptr; s->wave_bytes = 0; s->cap_paths = 0; s->wave_sets = 0;
	const size_t n = ((size_t)paths + 255u) & ~(size_t)255u;      /* every sub-array stays 256-byte aligned */
	const size_t per_set = n * (8u * 16u + 2u * 4u + 1u);         /* 137 B per path */
	const size_t bytes = per_set * (size_t)sets;
	void *base = nullptr;
	int rc = ctx_alloc(s->device, bytes, &base);
	if (rc) return rc;
	s->wave = base; s->wave_bytes = bytes;
	for (int k = 0; k < sets; ++k) {
		WaveBuffers &w = k ? s->wb2 : s->wb;
		uint8_t *q = static_cast<uint8_t *>(base) + per_set * (size_t)k;
		auto take = [&](size_t b) { uint8_t *r = q; q += b; return r; };
		w.stA[0] = (float4 *)take(n * 16); w.stA[1] = (float4 *)take(n * 16);
		w.stB[0] = (float4 *)take(n * 16); w.stB[1] = (float4 *)take(n * 16);
		w.stC[0] = (uint4 *)take(n * 16); w.stC[1] = (uint4 *)take(n * 16);
		w.hit = (float4 *)take(n * 16); w.L = (float4 *)take(n * 16);
		w.hitInst = (int *)take(n * 4); w.perm = (unsigned *)take(n * 4);
		w.hitKey = (unsigned char *)take(n);
	}
	s->cap_paths = paths;
	s->wave_sets = sets;
	return CRGPU_OK;
}

extern "C" int crgpu_scene_destroy(crgpu_scene *s) {
	if (!s) return CRGPU_OK;
	cudaSetDevice(s->device);
	if (s->stream) cudaStreamSynchronize(s->stream);
	if (s->own_stream && s->own_stream != s->stream) cudaStreamSynchronize(s->own_stream);
	if (s->stream2) cudaStreamSynchronize(s->stream2);
	ctx_free(s->device, s->slab, s->slab_bytes);
	ctx_free(s->device, s->wave, s->wave_bytes);
	ctx_free(s->device, s->small, s->small_bytes);
	ctx_free(s->device, s->fb, s->fb_floats * sizeof(float));
	ctx_free(s->device, s->fb8, s->fb_floats);
	ctx_free(s->device, s->pixels, s->pixel_cap * sizeof(uint32_t));
	for (cudaEvent_t e : s->ev) if (e) cudaEventDestroy(e);
	for (cudaEvent_t e : s->evAcc) if (e) cudaEventDestroy(e);
	if (s->evFork) cudaEventDestroy(s->evFork);
	if (s->stream2) cudaStreamDestroy(s->stream2);
	if (s->own_stream) cudaStreamDestroy(s->own_stream);
	delete s;
	return CRGPU_OK;
}

extern "C" void crgpu_prepared_free(crgpu_prepared *p) {
	if (!p) return;
	if (p->slab) { if (p->pinned) cudaFreeHost(p->slab); else free(p->slab); }
	delete p;
}
static int pfail(crgpu_prepared *p, int rc) { crgpu_prepared_free(p); return rc; }

extern "C" int crgpu_prepared_update_config(crgpu_prepared *p, const struct crs_scene *f) {
	if (!p || !f) return fail(CRGPU_ERR_BAD_ARGUMENT, "NULL argument");
	if (f->prefs.image_width == 0 || f->prefs.image_height == 0 || f->prefs.sample_count == 0)
		return fail(CRGPU_ERR_BAD_ARGUMENT, "empty image or zero samples");
	p->prefs = f->prefs;
	p->camera = f->camera;
	return CRGPU_OK;
}

extern "C" int crgpu_prepared_slab(const crgpu_prepared *p, const void **slab, size_t *bytes) {
	if (!p) return fail(CRGPU_ERR_BAD_ARGUMENT, "NULL argument");
	if (slab) *slab = p->slab;
	if (bytes) *bytes = p->slab_bytes;
	return CRGPU_OK;
}

extern "C" int crgpu_prepare(const struct crs_scene *f, crgpu_prepared **out) {
	if (!f || !out) return fail(CRGPU_ERR_BAD_ARGUMENT, "NULL argument");
	*out = nullptr;
	if (f->prefs.image_width == 0 || f->prefs.image_height == 0 || f->prefs.sample_count == 0)
		return fail(CRGPU_ERR_BAD_ARGUMENT, "empty image or zero samples");
	if (!node_ok(f, f->background) || f->nodes[f->background].kind != CRS_BSDF_BACKGROUND)
		return fail(CRGPU_ERR_UNSUPPORTED, "scene background must be a background node");
	if (f->top_bvh >= f->bvh_count) return fail(CRGPU_ERR_BAD_ARGUMENT, "top_bvh out of range");
	crgpu_prepared *p = new crgpu_prepared();
	p->slab = nullptr; p->pinned = false; p->slab_bytes = 0;
	p->prefs = f->prefs; p->camera = f->camera; p->background = f->background; p->instance_count = f->instance_count;
	p->xnodes = false;
	for (uint32_t i = 0; i < f->node_count; ++i) {
		const int k = f->nodes[i].kind;
		if (k == CRS_COLOR_VECTOCOLOR || k == CRS_COLOR_COMBINE_VALUE || k == CRS_COLOR_COMBINE_RGB || k == CRS_VALUE_MATH || k == CRS_VALUE_FRESNEL ||
			k == CRS_VALUE_RAYLENGTH || k == CRS_VECTOR_CONSTANT || k == CRS_VECTOR_NORMAL || k == CRS_VECTOR_VECMATH) p->xnodes = true;
	}
	p->texture_count = f->texture_count;
#define PFAIL(x) do { int rc_ = (x); if (rc_) return pfail(p, rc_); } while (0)

	/* materials + graph validation */
	std::vector<DevMaterial> mats(f->material_count);
	{
		bool uv = false;
		PFAIL(check_bsdf(f, f->background, 0, 0, &uv));
	}
	for (uint32_t i = 0; i < f->material_count; ++i) {
		const crs_material &m = f->materials[i];
		bool uv = false;
		PFAIL(check_bsdf(f, m.bsdf, 0, 0, &uv));
		DevMaterial d;
		memset(&d, 0, sizeof d);
		d.emission[0] = m.emission[0]; d.emission[1] = m.emission[1]; d.emission[2] = m.emission[2];
		d.IOR = m.IOR; d.bsdf = m.bsdf;
		/* x + w*0 == x bit-for-bit for finite w, so only non-zero (or non-finite) emission needs the add */
		const bool emits = !(m.emission[0] == 0.0f && m.emission[1] == 0.0f && m.emission[2] == 0.0f);
		d.flags = (uv ? 1u : 0u) | (emits ? 2u : 0u);
		mats[i] = d;
	}

	/* BVHs → pair nodes; triangles in leaf order; per-poly shading records.  The three products are independent once the
	 * slot offsets are known, and every element is computed from the flat scene alone, so they are filled by index on a
	 * few host threads (the upload bytes do not depend on the thread count).  This is most of crgpu_scene_create's time. */
	std::vector<PairNode> pairs;
	std::vector<DevBvh> bvhs(f->bvh_count);
	std::vector<PackedTri> tris;
	std::vector<uint32_t> slot_poly;
	std::vector<int32_t> top_prims;
	std::vector<uint32_t> mesh_of_bvh(f->bvh_count, 0xffffffffu);
	for (uint32_t m = 0; m < f->mesh_count; ++m) {
		if (f->meshes[m].bvh >= f->bvh_count) { return pfail(p, fail(CRGPU_ERR_BAD_ARGUMENT, "mesh bvh index out of range")); }
		mesh_of_bvh[f->meshes[m].bvh] = m;
	}
	std::vector<uint32_t> slot_off(f->bvh_count, 0u);      /* first triangle slot of every mesh BVH (0 for the top level) */
	uint64_t total_slots = 0;
	for (uint32_t b = 0; b < f->bvh_count; ++b) {
		const crs_bvh &src = f->bvhs[b];
		if ((uint64_t)src.node_offset + src.node_count > f->bvh_node_count || (uint64_t)src.prim_offset + src.prim_count > f->prim_index_count) {
			return pfail(p, fail(CRGPU_ERR_BAD_ARGUMENT, "bvh %u ranges out of bounds", b));
		}
		if (b == f->top_bvh) continue;
		if (mesh_of_bvh[b] == 0xffffffffu) { return pfail(p, fail(CRGPU_ERR_BAD_ARGUMENT, "bvh %u belongs to no mesh", b)); }
		slot_off[b] = (uint32_t)total_slots;
		total_slots += src.prim_count;
	}
	if (total_slots > 0xffffffffull) { return pfail(p, fail(CRGPU_ERR_UNSUPPORTED, "more than 2^32 triangle slots")); }
	for (uint32_t m = 0; m < f->mesh_count; ++m) {
		const crs_mesh &mesh = f->meshes[m];
		if ((uint64_t)mesh.poly_offset + mesh.poly_count > f->poly_count || (uint64_t)mesh.material_offset + mesh.material_count > f->material_count) {
			return pfail(p, fail(CRGPU_ERR_BAD_ARGUMENT, "mesh %u ranges out of bounds", m));
		}
	}
	tris.resize((size_t)total_slots);
	slot_poly.resize((size_t)total_slots);
	std::vector<ShadePoly> spolys(f->poly_count);
	HostError herr;

	/* (1) pair nodes of every BVH, in BVH order (sequential: each BVH appends behind the previous one) */
	std::thread pair_thread([&] {
		for (uint32_t b = 0; b < f->bvh_count; ++b) {
			const crs_bvh &src = f->bvhs[b];
			if (build_pairs(f, src, pairs, bvhs[b], b == f->top_bvh ? 0u : slot_off[b], &herr)) return;
			if (b != f->top_bvh) continue;
			for (uint32_t i = 0; i < src.prim_count; ++i) {
				const int32_t inst = f->prim_indices[src.prim_offset + i];
				if (inst < 0 || (uint32_t)inst >= f->instance_count) { herr.set(CRGPU_ERR_BAD_ARGUMENT, "top-level prim index out of range"); return; }
				top_prims.push_back(inst);
			}
		}
	});

	/* (2) triangles in leaf order */
	for (uint32_t b = 0; b < f->bvh_count; ++b) {
		if (b == f->top_bvh) continue;
		const crs_bvh &src = f->bvhs[b];
		const crs_mesh &mesh = f->meshes[mesh_of_bvh[b]];
		const uint32_t base = slot_off[b];
		host_parallel_for(src.prim_count, [&](uint32_t lo, uint32_t hi) {
			for (uint32_t i = lo; i < hi; ++i) {
				const int32_t local = f->prim_indices[src.prim_offset + i];
				if (local < 0 || (uint32_t)local >= mesh.poly_count) { herr.set(CRGPU_ERR_BAD_ARGUMENT, "prim index out of range"); return; }
				const uint32_t poly = mesh.poly_offset + (uint32_t)local;
				const crs_poly &p = f->polys[poly];
				for (int k = 0; k < 3; ++k)
					if (p.v[k] < 0 || (uint32_t)p.v[k] >= f->vertex_count) { herr.set(CRGPU_ERR_BAD_ARGUMENT, "vertex index out of range"); return; }
				float v0[3], v1[3], v2[3];
				f3(v0, f->vertices, (size_t)p.v[0]); f3(v1, f->vertices, (size_t)p.v[1]); f3(v2, f->vertices, (size_t)p.v[2]);
				PackedTri t;
				/* poly.c:20-22 — plain fp32 ops; this TU is compiled without contraction on the host side */
				for (int k = 0; k < 3; ++k) { t.v0[k] = v0[k]; t.e1[k] = v0[k] - v1[k]; t.e2[k] = v2[k] - v0[k]; }
				volatile float m0 = t.e1[1] * t.e2[2], m1 = t.e1[2] * t.e2[1], m2 = t.e1[2] * t.e2[0], m3 = t.e1[0] * t.e2[2],
							   m4 = t.e1[0] * t.e2[1], m5 = t.e1[1] * t.e2[0];
				t.n[0] = m0 - m1; t.n[1] = m2 - m3; t.n[2] = m4 - m5;
				tris[(size_t)base + i] = t;
				slot_poly[(size_t)base + i] = poly;
			}
		});
	}

	/* (3) per-poly shading records (meshes in order: should two meshes claim the same polygons, the later one wins as before) */
	for (uint32_t m = 0; m < f->mesh_count; ++m) {
		const crs_mesh &mesh = f->meshes[m];
		host_parallel_for(mesh.poly_count, [&](uint32_t lo, uint32_t hi) {
			for (uint32_t i = lo; i < hi; ++i) {
				const crs_poly &p = f->polys[mesh.poly_offset + i];
				ShadePoly sp;
				memset(&sp, 0, sizeof sp);
				bool has_n = p.has_normals != 0;
				for (int k = 0; k < 3 && has_n; ++k) if (p.n[k] < 0 || (uint32_t)p.n[k] >= f->normal_count) has_n = false;
				if (has_n) {
					f3(sp.n0, f->normals, (size_t)p.n[0]); f3(sp.n1, f->normals, (size_t)p.n[1]); f3(sp.n2, f->normals, (size_t)p.n[2]);
				} else if (p.has_normals) {
					herr.set(CRGPU_ERR_BAD_ARGUMENT, "normal index out of range"); return;
				} else {
					/* geometric normal e1 x e2 (poly.c:22,46), same operations as above */
					for (int k = 0; k < 3; ++k)
						if (p.v[k] < 0 || (uint32_t)p.v[k] >= f->vertex_count) { herr.set(CRGPU_ERR_BAD_ARGUMENT, "vertex index out of range"); return; }
					float v0[3], v1[3], v2[3], e1[3], e2[3];
					f3(v0, f->vertices, (size_t)p.v[0]); f3(v1, f->vertices, (size_t)p.v[1]); f3(v2, f->vertices, (size_t)p.v[2]);
					for (int k = 0; k < 3; ++k) { e1[k] = v0[k] - v1[k]; e2[k] = v2[k] - v0[k]; }
					volatile float m0 = e1[1] * e2[2], m1 = e1[2] * e2[1], m2 = e1[2] * e2[0], m3 = e1[0] * e2[2], m4 = e1[0] * e2[1], m5 = e1[1] * e2[0];
					sp.n0[0] = m0 - m1; sp.n0[1] = m2 - m3; sp.n0[2] = m4 - m5;
				}
				bool has_uv = mesh.texcoord_count != 0 && p.t[0] != -1;                          /* instance.c:151-153 */
				if (has_uv) {
					for (int k = 0; k < 3; ++k)
						if (p.t[k] < 0 || (uint32_t)p.t[k] >= f->texcoord_count) { herr.set(CRGPU_ERR_BAD_ARGUMENT, "texcoord index out of range"); return; }
					sp.t0[0] = f->texcoords[2 * (size_t)p.t[0]]; sp.t0[1] = f->texcoords[2 * (size_t)p.t[0] + 1];
					sp.t1[0] = f->texcoords[2 * (size_t)p.t[1]]; sp.t1[1] = f->texcoords[2 * (size_t)p.t[1] + 1];
					sp.t2[0] = f->texcoords[2 * (size_t)p.t[2]]; sp.t2[1] = f->texcoords[2 * (size_t)p.t[2] + 1];
				}
				if (p.material >= mesh.material_count) { herr.set(CRGPU_ERR_BAD_ARGUMENT, "poly material index out of range"); return; }
				sp.material = mesh.material_offset + p.material;
				sp.flags = (has_n ? 1u : 0u) | (has_uv ? 2u : 0u);
				spolys[mesh.poly_offset + i] = sp;
			}
		});
	}
	pair_thread.join();
	if (herr.code) { return pfail(p, fail(herr.code, "%s", herr.msg)); }

	/* instances */
	std::vector<DevInstance> insts(f->instance_count);
	for (uint32_t i = 0; i < f->instance_count; ++i) {
		const crs_instance &src = f->instances[i];
		DevInstance d;
		memset(&d, 0, sizeof d);
		memcpy(d.Ainv, src.Ainv, sizeof d.Ainv);
		memcpy(d.A, src.A, sizeof d.A);
		d.kind = src.kind;
		if (src.kind == CRS_INST_MESH) {
			if (src.object >= f->mesh_count) { return pfail(p, fail(CRGPU_ERR_BAD_ARGUMENT, "instance mesh index out of range")); }
			d.bvh = f->meshes[src.object].bvh;
			d.ray_offset = f->meshes[src.object].ray_offset;
		} else if (src.kind == CRS_INST_SPHERE) {
			if (src.object >= f->sphere_count) { return pfail(p, fail(CRGPU_ERR_BAD_ARGUMENT, "instance sphere index out of range")); }
			d.ray_offset = f->spheres[src.object].ray_offset;
			d.radius = f->spheres[src.object].radius;
			d.material = f->spheres[src.object].material;
			if (d.material >= f->material_count) { return pfail(p, fail(CRGPU_ERR_BAD_ARGUMENT, "sphere material out of range")); }
		} else { return pfail(p, fail(CRGPU_ERR_UNSUPPORTED, "instance kind %u (volumes are not reachable from the scene loader)", src.kind)); }
		insts[i] = d;
	}

	/* textures (data pointers are byte offsets into the texture section here; patched per device at upload) */
	std::vector<DevTexture> texs(f->texture_count);
	for (uint32_t i = 0; i < f->texture_count; ++i) {
		const crs_texture &t = f->textures[i];
		const uint64_t bytes = (uint64_t)t.width * t.height * t.channels * (t.is_float ? 4u : 1u);
		if (t.width == 0 || t.height == 0 || t.channels == 0 || t.channels > 4 || t.width > 65536u || t.height > 65536u ||
			t.data_offset > f->texdata_bytes || bytes > f->texdata_bytes - t.data_offset) {
			return pfail(p, fail(CRGPU_ERR_BAD_ARGUMENT, "texture %u malformed", i));
		}
		DevTexture d;
		d.width = t.width; d.height = t.height; d.channels = t.channels; d.is_float = t.is_float; d.has_alpha = t.has_alpha; d.pad = 0;
		d.wmask = (t.width & (t.width - 1u)) == 0u ? t.width - 1u : 0u;
		d.hmask = (t.height & (t.height - 1u)) == 0u ? t.height - 1u : 0u;
		d.data = reinterpret_cast<const uint8_t *>((uintptr_t)t.data_offset);
		texs[i] = d;
	}
	for (uint32_t i = 0; i < f->node_count; ++i)
		if (f->nodes[i].kind == CRS_COLOR_IMAGE && (f->nodes[i].tex >= (int32_t)f->texture_count || f->nodes[i].tex < -1))
			return pfail(p, fail(CRGPU_ERR_BAD_ARGUMENT, "node %u texture index out of range", i));

	std::vector<crs_node> nodes(f->nodes, f->nodes + f->node_count);

	p->top = bvhs[f->top_bvh];
	std::vector<float> lut(256);
	for (int i = 0; i < 256; ++i) { volatile float num = (float)i, den = 255.0f; lut[i] = num / den; }   /* IEEE divss == __fdiv_rn */

	/* lay the sections out in one slab (256-byte aligned each) and copy them in on the host threads */
	const void *src[SEC_COUNT] = { pairs.data(), tris.data(), slot_poly.data(), spolys.data(), top_prims.data(), bvhs.data(),
								   insts.data(), mats.data(), nodes.data(), texs.data(), lut.data(), f->texdata };
	const size_t len[SEC_COUNT] = { pairs.size() * sizeof(PairNode), tris.size() * sizeof(PackedTri),
									slot_poly.size() * sizeof(uint32_t), spolys.size() * sizeof(ShadePoly), top_prims.size() * sizeof(int32_t),
									bvhs.size() * sizeof(DevBvh), insts.size() * sizeof(DevInstance), mats.size() * sizeof(DevMaterial),
									nodes.size() * sizeof(crs_node), texs.size() * sizeof(DevTexture), lut.size() * sizeof(float), (size_t)f->texdata_bytes };
	size_t total = 0;
	for (int k = 0; k < SEC_COUNT; ++k) { p->off[k] = total; p->len[k] = len[k]; total += (len[k] + 255u) & ~(size_t)255u; }
	total += 512;                                                  /* room for the DevScene descriptor behind the arrays */
	p->slab_bytes = total;
	void *host = nullptr;
	if (cudaHostAlloc(&host, total, cudaHostAllocPortable) == cudaSuccess) p->pinned = true;
	else { cudaGetLastError(); host = malloc(total); p->pinned = false; }   /* no device yet (host-only tooling): pageable works, slower */
	if (!host) return pfail(p, fail(CRGPU_ERR_NOMEM, "cannot allocate the %zu-byte host slab", total));
	p->slab = static_cast<uint8_t *>(host);
	for (int k = 0; k < SEC_COUNT; ++k) {
		uint8_t *dst = p->slab + p->off[k];
		const uint8_t *from = static_cast<const uint8_t *>(src[k]);
		const size_t n = len[k];
		if (n) host_parallel_for((uint32_t)((n + 4095u) / 4096u), [&](uint32_t lo, uint32_t hi) {
			const size_t b0 = (size_t)lo * 4096u, b1 = (size_t)hi * 4096u < n ? (size_t)hi * 4096u : n;
			if (b1 > b0) memcpy(dst + b0, from + b0, b1 - b0);
		});
		memset(dst + n, 0, (((n + 255u) & ~(size_t)255u) - n));
	}
	memset(p->slab + total - 512, 0, 512);
#undef PFAIL
	*out = p;
	return CRGPU_OK;
}

extern "C" int crgpu_scene_create_prepared(const crgpu_prepared *p, int device, crgpu_scene **out) {
	if (!p || !out) return fail(CRGPU_ERR_BAD_ARGUMENT, "NULL argument");
	*out = nullptr;
	int ndev = 0;
	int rc = crgpu_device_count(&ndev);
	if (rc) return rc;
	if (device < 0 || device >= ndev) return fail(CRGPU_ERR_BAD_ARGUMENT, "device %d out of range (have %d)", device, ndev);
	CU(cudaSetDevice(device));

	crgpu_scene *s = new crgpu_scene();
	memset(&s->dev, 0, sizeof s->dev);
	memset(&s->wb, 0, sizeof s->wb);
	memset(&s->wb2, 0, sizeof s->wb2);
	s->wave_sets = 0; s->stream2 = nullptr; s->evAcc[0] = s->evAcc[1] = nullptr; s->evFork = nullptr;
	s->pixels = nullptr; s->pixel_cap = 0;
	s->device = device; s->xnodes = p->xnodes; s->dev_copy = nullptr; s->fb = nullptr; s->fb8 = nullptr; s->stream = nullptr; s->own_stream = nullptr; s->cap_paths = 0;
	s->slab = nullptr; s->slab_bytes = 0; s->small = nullptr; s->small_bytes = 0; s->wave = nullptr; s->wave_bytes = 0; s->fb_floats = 0;
	memset(s->fetched, 0, sizeof s->fetched);
	s->pend_paths = s->pend_launches = 0; s->pend_trace_ms = s->pend_shade_ms = s->pend_total_ms = 0.f;
	s->max_paths = 0;   /* set below from the free device memory */
	for (auto &e : s->ev) e = nullptr;
#define FAIL_IF(x) do { int rc_ = (x); if (rc_) { crgpu_scene_destroy(s); return rc_; } } while (0)
#define CUS(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { int rc_ = fail(CRGPU_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); crgpu_scene_destroy(s); return rc_; } } while (0)
	CUS(cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, device));
	CUS(cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking));
	s->stream = s->own_stream;
	for (auto &e : s->ev) CUS(cudaEventCreate(&e));
	CUS(cudaStreamCreateWithFlags(&s->stream2, cudaStreamNonBlocking));
	for (auto &e : s->evAcc) CUS(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
	CUS(cudaEventCreateWithFlags(&s->evFork, cudaEventDisableTiming));

	/* the scene: one block, one copy */
	FAIL_IF(ctx_alloc(device, p->slab_bytes, &s->slab));
	s->slab_bytes = p->slab_bytes;
	uint8_t *base = static_cast<uint8_t *>(s->slab);
	CUS(cudaMemcpyAsync(base, p->slab, p->slab_bytes, cudaMemcpyHostToDevice, s->stream));
	if (p->texture_count) {                 /* texture table with this device's addresses */
		std::vector<DevTexture> texs(p->texture_count);
		memcpy(texs.data(), p->slab + p->off[SEC_TEXS], p->texture_count * sizeof(DevTexture));
		for (DevTexture &t : texs) t.data = base + p->off[SEC_TEXDATA] + (uintptr_t)t.data;
		CUS(cudaMemcpyAsync(base + p->off[SEC_TEXS], texs.data(), texs.size() * sizeof(DevTexture), cudaMemcpyHostToDevice, s->stream));
		CUS(cudaStreamSynchronize(s->stream));   /* texs is a local pageable buffer */
	}
	DevScene &d = s->dev;
	d.cam.sensor_x = p->camera.sensor_x; d.cam.sensor_y = p->camera.sensor_y;
	d.cam.aperture = p->camera.aperture; d.cam.focal_distance = p->camera.focal_distance;
	memcpy(d.cam.forward, p->camera.forward, 12); memcpy(d.cam.right, p->camera.right, 12); memcpy(d.cam.up, p->camera.up, 12);
	d.cam.width = p->camera.width; d.cam.height = p->camera.height;
	memcpy(d.cam.A, p->camera.A, sizeof d.cam.A);
	d.image_width = p->prefs.image_width; d.image_height = p->prefs.image_height;
	d.sample_count = p->prefs.sample_count; d.bounces = p->prefs.bounces;
	d.background = p->background;
	d.instance_count = p->instance_count;
	d.top = p->top;
	d.pairs = reinterpret_cast<const PairNode *>(base + p->off[SEC_PAIRS]);
	d.tris = reinterpret_cast<const PackedTri *>(base + p->off[SEC_TRIS]);
	d.slot_poly = reinterpret_cast<const uint32_t *>(base + p->off[SEC_SLOT_POLY]);
	d.spolys = reinterpret_cast<const ShadePoly *>(base + p->off[SEC_SPOLYS]);
	d.top_prims = reinterpret_cast<const int32_t *>(base + p->off[SEC_TOP_PRIMS]);
	d.bvhs = reinterpret_cast<const DevBvh *>(base + p->off[SEC_BVHS]);
	d.instances = reinterpret_cast<const DevInstance *>(base + p->off[SEC_INSTS]);
	d.materials = reinterpret_cast<const DevMaterial *>(base + p->off[SEC_MATS]);
	d.nodes = reinterpret_cast<const crs_node *>(base + p->off[SEC_NODES]);
	d.textures = reinterpret_cast<const DevTexture *>(base + p->off[SEC_TEXS]);
	d.u8_to_unit = reinterpret_cast<const float *>(base + p->off[SEC_LUT]);
	static_assert(sizeof(DevScene) <= 512, "DevScene must fit the descriptor slot behind the scene arrays");
	s->dev_copy = reinterpret_cast<DevScene *>(base + p->slab_bytes - 512);
	CUS(cudaMemcpyAsync(s->dev_copy, &s->dev, sizeof(DevScene), cudaMemcpyHostToDevice, s->stream));

	s->fb_floats = (size_t)d.image_width * d.image_height * 3u;
	{ void *q = nullptr; FAIL_IF(ctx_alloc(device, s->fb_floats * sizeof(float), &q)); s->fb = static_cast<float *>(q); }
	CUS(cudaMemsetAsync(s->fb, 0, s->fb_floats * sizeof(float), s->stream));
	{	/* per wave set: hist[512] + counts[64]; then the shared stats[80] */
		const size_t set_bytes = 512 * sizeof(unsigned) + 256;
		s->small_bytes = 2 * set_bytes + 80 * sizeof(unsigned long long);
		FAIL_IF(ctx_alloc(device, s->small_bytes, &s->small));
		CUS(cudaMemsetAsync(s->small, 0, s->small_bytes, s->stream));
		uint8_t *sm = static_cast<uint8_t *>(s->small);
		s->wb.hist = reinterpret_cast<unsigned *>(sm);
		s->wb.counts = s->wb.hist + 512;
		s->wb2.hist = reinterpret_cast<unsigned *>(sm + set_bytes);
		s->wb2.counts = s->wb2.hist + 512;
		s->wb.stats = s->wb2.stats = reinterpret_cast<unsigned long long *>(sm + 2 * set_bytes);
	}
	{
		/* Paths in flight per wavefront batch.  Every batch pays a fixed ~7 ms (the serial chain of its bounces: each
		 * late bounce lasts as long as its slowest ray), so batches should be as large as memory allows:
		 * 137 B of wavefront state per path; use at most 40% of the free HBM (cached blocks count as free), capped at 256M paths. */
		size_t free_b = 0, total_b = 0;
		CUS(cudaMemGetInfo(&free_b, &total_b));
		free_b += ctx_cached_bytes(device);
		uint64_t fit = (uint64_t)((double)free_b * 0.40 / 137.0);
		if (fit > (256ull << 20)) fit = 256ull << 20;
		if (fit < (1ull << 20)) fit = 1ull << 20;
		s->max_paths = fit;
	}
	CUS(cudaStreamSynchronize(s->stream));
#undef FAIL_IF
#undef CUS
	*out = s;
	return CRGPU_OK;
}

extern "C" int crgpu_scene_create(const struct crs_scene *f, int device, crgpu_scene **out) {
	if (!f || !out) return fail(CRGPU_ERR_BAD_ARGUMENT, "NULL argument");
	*out = nullptr;
	int ndev = 0;
	int rc = crgpu_device_count(&ndev);
	if (rc) return rc;
	if (device < 0 || device >= ndev) return fail(CRGPU_ERR_BAD_ARGUMENT, "device %d out of range (have %d)", device, ndev);
	CU(cudaSetDevice(device));
	crgpu_prepared *p = nullptr;
	rc = crgpu_prepare(f, &p);
	if (rc) return rc;
	rc = crgpu_scene_create_prepared(p, device, out);
	crgpu_prepared_free(p);
	return rc;
}

extern "C" int crgpu_set_max_paths_in_flight(crgpu_scene *s, uint64_t max_paths) {
	if (!s || max_paths < 1024) return fail(CRGPU_ERR_BAD_ARGUMENT, "max_paths must be >= 1024");
	if (max_paths > (1ull << 31)) return fail(CRGPU_ERR_BAD_ARGUMENT, "max_paths must be <= 2^31");
	s->max_paths = max_paths;
	return CRGPU_OK;
}

static int check_rect(const crgpu_scene *s, int x0, int y0, int x1, int y1) {
	if (x0 < 0 || y0 < 0 || x1 > (int)s->dev.image_width || y1 > (int)s->dev.image_height || x1 <= x0 || y1 <= y0)
		return fail(CRGPU_ERR_BAD_ARGUMENT, "tile [%d,%d)x[%d,%d) outside the %ux%u image", x0, x1, y0, y1, s->dev.image_width, s->dev.image_height);
	return CRGPU_OK;
}

/* the wavefront driver: passes [pass_begin, +pass_count) over a pixel set (a rectangle, or an explicit list) */
static int render_pixels(crgpu_scene *s, TileDesc base, uint64_t tile_pixels, int pass_begin, int pass_count,
						 unsigned flags, struct crgpu_stats *stats) {
	if (pass_begin < 0 || pass_count < 0 || (uint64_t)pass_begin + (uint64_t)pass_count > s->dev.sample_count)
		return fail(CRGPU_ERR_BAD_ARGUMENT, "passes [%d,%d) outside [0,%u)", pass_begin, pass_begin + pass_count, s->dev.sample_count);
	if (tile_pixels > s->max_paths) {
		/* more pixels than paths in flight: walk the pixel set in pieces (rows of the rectangle / ranges of the list) */
		const unsigned inner = flags | CRGPU_FLAG_ASYNC;
		if (base.pixels) {
			for (uint64_t p0 = 0; p0 < tile_pixels; p0 += s->max_paths) {
				TileDesc part = base;
				part.pixels = base.pixels + p0;
				const uint64_t cnt = tile_pixels - p0 < s->max_paths ? tile_pixels - p0 : s->max_paths;
				int rc = render_pixels(s, part, cnt, pass_begin, pass_count, inner, nullptr);
				if (rc) return rc;
			}
		} else {
			const uint64_t rows = s->max_paths / (uint64_t)base.tw;
			if (rows < 1) return fail(CRGPU_ERR_BAD_ARGUMENT, "tile is %d pixels wide > max paths in flight %llu", base.tw, (unsigned long long)s->max_paths);
			for (int y = 0; y < base.th; y += (int)rows) {
				TileDesc part = base;
				part.y0 = base.y0 + y;
				part.th = base.th - y < (int)rows ? base.th - y : (int)rows;
				int rc = render_pixels(s, part, (uint64_t)part.tw * (uint64_t)part.th, pass_begin, pass_count, inner, nullptr);
				if (rc) return rc;
			}
		}
		if (flags & CRGPU_FLAG_ASYNC) return CRGPU_OK;
		return crgpu_get_stats(s, stats);
	}
	if (pass_count == 0 || tile_pixels == 0) {          /* an empty pass range is a no-op (and must not reach the batch arithmetic below) */
		if (flags & CRGPU_FLAG_ASYNC) return CRGPU_OK;
		return crgpu_get_stats(s, stats);
	}
	const bool count = (flags & CRGPU_FLAG_COUNT) != 0;
	const bool timing = (flags & CRGPU_FLAG_TIME_KERNELS) != 0;
	/* Batches.  A batch pays a fixed cost of several ms: its bounces 5..12 hold too few rays to fill 148 SMs, and every bounce lasts
	 * as long as its slowest ray.  So (1) batches are as large as the path budget allows and of EQUAL size (a 987 + 13 split wastes
	 * a whole tail on 13 passes), and (2) with two or more batches the budget is split into two wave sets that run on two streams:
	 * the thin tail of one batch overlaps the fat first bounces of the next.  Only the accumulate step is ordered (the running
	 * average is taken in pass order, renderer.c:288-291): batch b's k_accumulate waits for batch b-1's. */
	uint64_t batch = s->max_paths / tile_pixels;
	if (batch < 1) batch = 1;
	int sets = 1;
	if (!timing && !count && batch < (uint64_t)pass_count && batch >= 2) { sets = 2; batch /= 2; }
	if (batch > (uint64_t)pass_count) batch = (uint64_t)pass_count;
	{
		const uint64_t nb = ((uint64_t)pass_count + batch - 1) / batch;
		if (nb > 0) batch = ((uint64_t)pass_count + nb - 1) / nb;   /* equal shares */
		if (batch < 1) batch = 1;
	}
	int rc = alloc_wave(s, tile_pixels * batch, sets);
	if (rc) return rc;

	const int maxDepth = (int)s->dev.bounces;
	const int grid = s->sm_count * 8;
	uint64_t launches = 0;
	float trace_ms = 0.f, shade_ms = 0.f;
	if (timing) CU(cudaEventRecord(s->ev[0], s->stream));
	std::vector<cudaEvent_t> tev;   /* per-kernel events when timing */
	if (sets == 2) {                /* fork: the second stream starts behind whatever is queued on the first */
		CU(cudaEventRecord(s->evFork, s->stream));
		CU(cudaStreamWaitEvent(s->stream2, s->evFork, 0));
	}
	int bi = 0;
	for (int pb = pass_begin; pb < pass_begin + pass_count; pb += (int)batch, ++bi) {
		const int set = sets == 2 ? (bi & 1) : 0;
		cudaStream_t st = set ? s->stream2 : s->stream;
		const WaveBuffers &wb = set ? s->wb2 : s->wb;
		TileDesc td = base;
		td.npix = (unsigned)tile_pixels;
		td.pass_begin = pb;
		td.pass_count = (pass_begin + pass_count - pb) < (int)batch ? (pass_begin + pass_count - pb) : (int)batch;
		crg_launch_generate(s->dev, wb, td, grid, st); ++launches;
		/* bounces == 0: pathTrace's loop never runs and every sample is black (pathtrace.c:34-36,59).  L is write-once by
		 * design (cr_add_radiance / cr_finish_path), so with no bounce nothing would write it: clear it here instead */
		if (maxDepth == 0) CU(cudaMemsetAsync(wb.L, 0, (size_t)tile_pixels * (size_t)td.pass_count * sizeof(float4), st));
		int cur = 0;
		for (int depth = 0; depth < maxDepth; ++depth) {
			if (depth >= CRG_TAIL_FROM && !count) { crg_launch_tail(s->dev_copy, wb, cur, depth, maxDepth, s->xnodes, st); ++launches; }
			if (timing) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); tev.push_back(e); }
			crg_launch_trace(s->dev, wb, cur, count, st);
			if (timing) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); tev.push_back(e); }
			crg_launch_bucket(wb, cur, grid, st);
			crg_launch_shade(s->dev_copy, wb, cur, depth, maxDepth, s->xnodes, grid, st);
			if (timing) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); tev.push_back(e); }
			launches += 4;                                                       /* K2, K4, K3 miss half, K3 hit half */
			cur ^= 1;
		}
		if (sets == 2 && bi > 0) CU(cudaStreamWaitEvent(st, s->evAcc[set ^ 1], 0));      /* pass order of the running average */
		crg_launch_accumulate(s->fb, wb.L, td, (int)s->dev.image_width, (int)s->dev.image_height, grid, st); ++launches;
		if (sets == 2) CU(cudaEventRecord(s->evAcc[set], st));
	}
	if (sets == 2 && bi > 0) {      /* join: everything queued later on the scene's stream comes after both */
		CU(cudaStreamWaitEvent(s->stream, s->evAcc[(bi - 1) & 1], 0));
		if (bi > 1) CU(cudaStreamWaitEvent(s->stream, s->evAcc[bi & 1], 0));
	}
	cudaStream_t st = s->stream;
	if (timing) CU(cudaEventRecord(s->ev[1], st));
	CU(cudaGetLastError());
	s->pend_paths += tile_pixels * (uint64_t)pass_count;
	s->pend_launches += launches;
	if (timing) {
		CU(cudaStreamSynchronize(st));
		float total_ms = 0.f;
		cudaEventElapsedTime(&total_ms, s->ev[0], s->ev[1]);
		for (size_t i = 0; i + 3 <= tev.size(); i += 3) {
			float a = 0.f, b = 0.f;
			cudaEventElapsedTime(&a, tev[i], tev[i + 1]);
			cudaEventElapsedTime(&b, tev[i + 1], tev[i + 2]);
			trace_ms += a; shade_ms += b;
		}
		for (cudaEvent_t e : tev) cudaEventDestroy(e);
		s->pend_trace_ms += trace_ms; s->pend_shade_ms += shade_ms; s->pend_total_ms += total_ms;
	}
	if (flags & CRGPU_FLAG_ASYNC) return CRGPU_OK;
	return crgpu_get_stats(s, stats);
}

extern "C" int crgpu_render_tile(crgpu_scene *s, int x0, int y0, int x1, int y1, int pass_begin, int pass_count,
								 unsigned flags, struct crgpu_stats *stats) {
	if (!s) return fail(CRGPU_ERR_BAD_ARGUMENT, "scene is NULL");
	int rc = check_rect(s, x0, y0, x1, y1);
	if (rc) return rc;
	CU(cudaSetDevice(s->device));
	TileDesc td;
	memset(&td, 0, sizeof td);
	td.x0 = x0; td.y0 = y0; td.tw = x1 - x0; td.th = y1 - y0;
	td.pixels = nullptr;
	return render_pixels(s, td, (uint64_t)td.tw * (uint64_t)td.th, pass_begin, pass_count, flags, stats);
}

extern "C" int crgpu_render_tiles(crgpu_scene *s, const int *rects, int nrects, int pass_begin, int pass_count,
								  unsigned flags, struct crgpu_stats *stats) {
	if (!s || !rects || nrects < 1) return fail(CRGPU_ERR_BAD_ARGUMENT, "bad tile list");
	if (s->dev.image_width > 65535u || s->dev.image_height > 65535u) return fail(CRGPU_ERR_UNSUPPORTED, "tile lists need image dimensions <= 65535");
	CU(cudaSetDevice(s->device));
	uint64_t total = 0;
	for (int i = 0; i < nrects; ++i) {
		int rc = check_rect(s, rects[4 * i], rects[4 * i + 1], rects[4 * i + 2], rects[4 * i + 3]);
		if (rc) return rc;
		total += (uint64_t)(rects[4 * i + 2] - rects[4 * i]) * (uint64_t)(rects[4 * i + 3] - rects[4 * i + 1]);
	}
	std::vector<int> key(rects, rects + 4 * (size_t)nrects);
	if (key != s->pixel_key) {                         /* rebuild the pixel list only when the tile set changes */
		if (total > 0xffffffffull) return fail(CRGPU_ERR_UNSUPPORTED, "tile set of more than 2^32 pixels");
		/* the list is expanded ON THE DEVICE from the rectangles (a 1080p frame is 2 M entries, an 8K frame 33 M: building and
		 * uploading them from the host cost ~10 ms per frame): upload 16 B + 4 B per tile, one kernel writes x | y << 16 */
		std::vector<unsigned> offs((size_t)nrects);
		unsigned acc = 0u;
		for (int i = 0; i < nrects; ++i) { offs[(size_t)i] = acc; acc += (unsigned)((rects[4 * i + 2] - rects[4 * i]) * (rects[4 * i + 3] - rects[4 * i + 1])); }
		const size_t need = (size_t)total * sizeof(uint32_t) + (size_t)nrects * 20u + 256u;
		if (s->pixel_cap * sizeof(uint32_t) < need) {
			CU(cudaStreamSynchronize(s->stream));       /* the previous list may still be in use by queued kernels */
			ctx_free(s->device, s->pixels, s->pixel_cap * sizeof(uint32_t));
			s->pixels = nullptr; s->pixel_cap = 0;
			void *q = nullptr;
			int arc = ctx_alloc(s->device, need, &q);
			if (arc) return arc;
			s->pixels = static_cast<uint32_t *>(q);
			s->pixel_cap = (need + 3u) / 4u;
		}
		/* rectangle table behind the pixel list (same block); both copies are from pageable memory, i.e. staged before the call
		 * returns, and ordered before the kernel on the scene's stream */
		uint8_t *tab = reinterpret_cast<uint8_t *>(s->pixels) + (((size_t)total * sizeof(uint32_t) + 255u) & ~(size_t)255u);
		CU(cudaMemcpyAsync(tab, rects, (size_t)nrects * 16u, cudaMemcpyHostToDevice, s->stream));
		CU(cudaMemcpyAsync(tab + (size_t)nrects * 16u, offs.data(), (size_t)nrects * 4u, cudaMemcpyHostToDevice, s->stream));
		CU(cudaStreamSynchronize(s->stream));           /* offs is a local; costs ~20 us, once per tile set */
		crg_launch_pixel_list(s->pixels, reinterpret_cast<const int4 *>(tab), reinterpret_cast<const unsigned *>(tab + (size_t)nrects * 16u), nrects, s->stream);
		CU(cudaGetLastError());
		s->pixel_key.swap(key);
	}
	TileDesc td;
	memset(&td, 0, sizeof td);
	td.pixels = s->pixels;
	return render_pixels(s, td, total, pass_begin, pass_count, flags, stats);
}

extern "C" int crgpu_get_stats(crgpu_scene *s, struct crgpu_stats *stats) {
	if (!s) return fail(CRGPU_ERR_BAD_ARGUMENT, "scene is NULL");
	CU(cudaSetDevice(s->device));
	unsigned long long h[8];
	CU(cudaMemcpyAsync(h, s->wb.stats, sizeof h, cudaMemcpyDeviceToHost, s->stream));
	CU(cudaStreamSynchronize(s->stream));
	if (h[7] != s->fetched[7]) {
		memcpy(s->fetched, h, sizeof h);
		return fail(CRGPU_ERR_CUDA, "traversal watchdog: %llu ray(s) exceeded the step limit (corrupt BVH?)", h[7]);
	}
	if (stats) {
		memset(stats, 0, sizeof *stats);
		stats->paths = s->pend_paths;
		stats->rays = h[0] - s->fetched[0]; stats->node_pairs = h[1] - s->fetched[1]; stats->tri_tests = h[2] - s->fetched[2];
		stats->sphere_tests = h[3] - s->fetched[3]; stats->inst_visits = h[4] - s->fetched[4];
		stats->kernel_launches = s->pend_launches;
		stats->trace_ms = s->pend_trace_ms; stats->shade_ms = s->pend_shade_ms; stats->total_ms = s->pend_total_ms;
	}
	memcpy(s->fetched, h, sizeof h);
	s->pend_paths = s->pend_launches = 0; s->pend_trace_ms = s->pend_shade_ms = s->pend_total_ms = 0.f;
	return CRGPU_OK;
}

extern "C" int crgpu_set_stream(crgpu_scene *s, void *cuda_stream) {
	if (!s) return fail(CRGPU_ERR_BAD_ARGUMENT, "scene is NULL");
	CU(cudaSetDevice(s->device));
	CU(cudaStreamSynchronize(s->stream));
	s->stream = static_cast<cudaStream_t>(cuda_stream);      /* NULL is a valid handle: the legacy default stream */
	return CRGPU_OK;
}

extern "C" int crgpu_use_own_stream(crgpu_scene *s) {
	if (!s) return fail(CRGPU_ERR_BAD_ARGUMENT, "scene is NULL");
	CU(cudaSetDevice(s->device));
	CU(cudaStreamSynchronize(s->stream));
	s->stream = s->own_stream;
	return CRGPU_OK;
}

extern "C" int crgpu_framebuffer_clear(crgpu_scene *s) {
	if (!s) return fail(CRGPU_ERR_BAD_ARGUMENT, "scene is NULL");
	CU(cudaSetDevice(s->device));
	CU(cudaMemsetAsync(s->fb, 0, s->fb_floats * sizeof(float), s->stream));
	CU(cudaStreamSynchronize(s->stream));
	return CRGPU_OK;
}

static int fb_copy(crgpu_scene *s, float *host, int x0, int y0, int x1, int y1, bool to_host) {
	if (!s || !host) return fail(CRGPU_ERR_BAD_ARGUMENT, "NULL argument");
	CU(cudaSetDevice(s->device));
	const size_t W = s->dev.image_width, H = s->dev.image_height;
	if (x1 <= x0) { x0 = 0; y0 = 0; x1 = (int)W; y1 = (int)H; }
	int rc = check_rect(s, x0, y0, x1, y1);
	if (rc) return rc;
	/* rows y0..y1-1 (y up) are storage rows H-y1 .. H-1-y0 */
	const size_t row0 = H - (size_t)y1, rows = (size_t)(y1 - y0);
	const size_t off = (row0 * W + (size_t)x0) * 3u;
	const size_t pitch = W * 3u * sizeof(float), width = (size_t)(x1 - x0) * 3u * sizeof(float);
	if (to_host) CU(cudaMemcpy2DAsync(host + off, pitch, s->fb + off, pitch, width, rows, cudaMemcpyDeviceToHost, s->stream));
	else CU(cudaMemcpy2DAsync(s->fb + off, pitch, host + off, pitch, width, rows, cudaMemcpyHostToDevice, s->stream));
	CU(cudaStreamSynchronize(s->stream));
	return CRGPU_OK;
}
extern "C" int crgpu_framebuffer_read(crgpu_scene *s, float *host_rgb, int x0, int y0, int x1, int y1) {
	return fb_copy(s, host_rgb, x0, y0, x1, y1, true);
}
extern "C" int crgpu_framebuffer_write(crgpu_scene *s, const float *host_rgb, int x0, int y0, int x1, int y1) {
	return fb_copy(s, const_cast<float *>(host_rgb), x0, y0, x1, y1, false);
}

extern "C" int crgpu_framebuffer_to_srgb8(crgpu_scene *s, uint8_t *host_rgb8) {
	if (!s || !host_rgb8) return fail(CRGPU_ERR_BAD_ARGUMENT, "NULL argument");
	CU(cudaSetDevice(s->device));
	if (!s->fb8) { void *q = nullptr; int arc = ctx_alloc(s->device, s->fb_floats, &q); if (arc) return arc; s->fb8 = static_cast<uint8_t *>(q); }
	crg_launch_to_srgb8(s->fb, s->fb8, s->fb_floats, s->sm_count * 8, s->stream);
	CU(cudaGetLastError());
	CU(cudaMemcpyAsync(host_rgb8, s->fb8, s->fb_floats, cudaMemcpyDeviceToHost, s->stream));
	CU(cudaStreamSynchronize(s->stream));
	return CRGPU_OK;
}

extern "C" int crgpu_framebuffer_device_ptr(crgpu_scene *s, void **dev_ptr, size_t *bytes) {
	if (!s || !dev_ptr) return fail(CRGPU_ERR_BAD_ARGUMENT, "NULL argument");
	*dev_ptr = s->fb;
	if (bytes) *bytes = s->fb_floats * sizeof(float);
	return CRGPU_OK;
}

extern "C" int crgpu_scene_info(crgpu_scene *s, int *device, int *width, int *height) {
	if (!s) return fail(CRGPU_ERR_BAD_ARGUMENT, "scene is NULL");
	if (device) *device = s->device;
	if (width) *width = (int)s->dev.image_width;
	if (height) *height = (int)s->dev.image_height;
	return CRGPU_OK;
}

extern "C" int crgpu_trace_kat(crgpu_scene *s, const int32_t *xyp, int count, void *records_out) {
	if (!s || !xyp || !records_out || count < 0) return fail(CRGPU_ERR_BAD_ARGUMENT, "bad argument");
	if (count == 0) return CRGPU_OK;
	CU(cudaSetDevice(s->device));
	int32_t *dx = nullptr;
	void *dk = nullptr;
	CU(cudaMalloc((void **)&dx, (size_t)count * 3 * sizeof(int32_t)));
	CU(cudaMalloc((void **)&dk, (size_t)count * CRG_HITKAT_BYTES));
	CU(cudaMemcpyAsync(dx, xyp, (size_t)count * 3 * sizeof(int32_t), cudaMemcpyHostToDevice, s->stream));
	crg_launch_kat(s->dev_copy, dx, count, dk, s->stream);
	cudaError_t e = cudaGetLastError();
	if (e == cudaSuccess) e = cudaMemcpyAsync(records_out, dk, (size_t)count * CRG_HITKAT_BYTES, cudaMemcpyDeviceToHost, s->stream);
	if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
	cudaFree(dx); cudaFree(dk);
	if (e != cudaSuccess) return fail(CRGPU_ERR_CUDA, "trace_kat: %s", cudaGetErrorString(e));
	return CRGPU_OK;
}

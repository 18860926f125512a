/*
 * crgpu_trace.cu — K1 (primary-ray generation) and K2 (two-level BVH traversal): see crgpu_wave.cuh.
 * Everything here is force-inlined; the scene descriptor travels as a by-value kernel parameter so
 * its pointers sit in the constant bank.
 */
#include <mutex>
#include "crgpu_wave.cuh"
#include "crgpu_trace.cuh"

/* ---- pixel list of a tile set: blockIdx.y = tile, the block's threads walk its pixels row by row (crgpu_render_tiles) ---------------- */
__global__ void __launch_bounds__(256) k_pixel_list(uint32_t *__restrict__ pixels, const int4 *__restrict__ rects, const unsigned *__restrict__ offs) {
	const int4 r = rects[blockIdx.y];
	const unsigned w = (unsigned)(r.z - r.x), n = w * (unsigned)(r.w - r.y);
	uint32_t *out = pixels + offs[blockIdx.y];
	for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const unsigned y = i / w, x = i - y * w;
		out[i] = (uint32_t)(r.x + (int)x) | ((uint32_t)(r.y + (int)y) << 16);
	}
}
void crg_launch_pixel_list(uint32_t *pixels, const int4 *rects, const unsigned *offs, int nrects, cudaStream_t st) {
	for (int first = 0; first < nrects; first += 32768) {            /* gridDim.y <= 65535 */
		const int cnt = nrects - first < 32768 ? nrects - first : 32768;
		k_pixel_list<<<dim3(4, (unsigned)cnt), 256, 0, st>>>(pixels, rects + first, offs + first);
	}
}

/* ---- K1 ------------------------------------------------------------------------------------------------------------ */
__global__ void __launch_bounds__(256) k_generate(DevScene sc, WaveBuffers wb, TileDesc td) {
	const unsigned tile_pixels = td.npix;
	const unsigned n = tile_pixels * (unsigned)td.pass_count;
	for (unsigned id = blockIdx.x * blockDim.x + threadIdx.x; id < n; id += gridDim.x * blockDim.x) {
		const unsigned pl = id / tile_pixels, px = id - pl * tile_pixels;
		int x, y;
		crg_pixel_xy(td, px, x, y);
		const uint32_t pixIdx = (uint32_t)(y * (int)sc.image_width + x);                        /* renderer.c:280 */
		uint64_t rng = cr_rng_init(pixIdx, (uint32_t)(td.pass_begin + (int)pl), sc.sample_count);
		v3 o, d;
		cr_camera_ray(sc.cam, x, y, rng, o, d);
		wb.stA[0][id] = make_float4(o.x, o.y, o.z, d.x);
		wb.stB[0][id] = make_float4(d.y, d.z, 1.0f, 1.0f);
		wb.stC[0][id] = make_uint4(__float_as_uint(1.0f), id, (unsigned)(rng & 0xffffffffull), (unsigned)(rng >> 32));
	}
	if (blockIdx.x == 0 && threadIdx.x == 0) { wb.counts[0] = n; wb.counts[1] = 0u; wb.counts[2] = 0u; wb.counts[3] = 0u; }
	if (blockIdx.x == 0) { for (int k = 0; k < 2; ++k) wb.hist[k * 256 + threadIdx.x] = 0u; }   /* blockDim.x == 256 */
}

/* ---- K2: persistent warps with dynamic ray refill ----------------------------------------------------------------------
 * Ray lengths vary a lot (hdr.json: 7 child-pair steps on average, >200 for some), so a warp that takes 32
 * rays and waits for the slowest one idles most lanes (ncu: 7-10 active threads/warp).  Here every warp keeps
 * its 32 traversal state machines in registers and, whenever fewer than CRG_REFILL lanes are busy, pulls new
 * rays for the idle lanes from a global work counter (one ballot + one atomicAdd per refill, indices handed
 * out in lane order so neighbouring lanes still get neighbouring — coherent — rays). */
#define CRG_REFILL 16
#define CRG_NODE_BURST 3
#define CRG_INST_MIN 8
#define CRG_MAX_STEPS 8000000u   /* > 30x the node count of any scene that fits the 2^23-node address space we support */

template <bool COUNT>
__global__ void __launch_bounds__(256, 3) k_trace(DevScene sc, WaveBuffers wb, int cur) {
	const unsigned n = wb.counts[cur];
	const unsigned lane = threadIdx.x & 31u;
	const float4 *__restrict__ stA = wb.stA[cur];
	const float4 *__restrict__ stB = wb.stB[cur];
	TraceCounters tc = { 0u, 0u, 0u, 0u };
	__shared__ unsigned s_hist[256];
	s_hist[threadIdx.x] = 0u;            /* blockDim.x == 256 */
	__syncthreads();
	uint32_t stack[2 * CRG_MAX_STACK + 2];
	Traversal<COUNT> tr;
	tr.stack = stack;
	tr.begin(sc, v3make(0.f, 0.f, 0.f), v3make(0.f, 0.f, 1.f));   /* every lane holds a VALID (idle) state from the start */
	bool busy = false;
	bool exhausted = false;          /* warp-uniform: the work counter ran past n */
	unsigned ray = 0u;
	unsigned steps = 0u;             /* safety net: a lane that exceeds CRG_MAX_STEPS is abandoned and flagged */
	while (true) {
		unsigned active = __ballot_sync(0xffffffffu, busy);
		if (!exhausted && __popc(active) < CRG_REFILL) {
			const unsigned idle = ~active;
			const unsigned nidle = (unsigned)__popc(idle);
			unsigned base = 0u;
			if (lane == 0u) base = atomicAdd(&wb.counts[2], nidle);
			base = __shfl_sync(0xffffffffu, base, 0);
			if (base + nidle >= n) exhausted = true;
			const unsigned slot = base + (unsigned)__popc(idle & ((1u << lane) - 1u));
			if (!busy && slot < n) {
				const float4 a = stA[slot];
				const float4 b = stB[slot];
				ray = slot;
				steps = 0u;
				tr.begin(sc, v3make(a.x, a.y, a.z), v3make(a.w, b.x, b.y));
				busy = true;
			}
			active = __ballot_sync(0xffffffffu, busy);
		}
		if (active == 0u) break;         /* nothing in flight and nothing left to fetch */
		/* Phase N: up to CRG_NODE_BURST child-pair steps for every lane that is inside a BVH.  Lanes that reach a
		 * top-level leaf (instance work) or finish wait here, so that the instance / write-back code below runs
		 * for many lanes at once instead of being serialised against node steps in every iteration. */
#pragma unroll 1
		for (int k = 0; k < CRG_NODE_BURST; ++k) {
			const bool wn = busy && tr.wants_node();
			if (!__any_sync(0xffffffffu, wn)) break;
			if (wn) { tr.node_step(sc, &tc); ++steps; }
		}
		/* Phase I: one pending instance (ray transform + sphere test, or entry into a mesh BVH).  ncu (profiles/r01: 19.8% of K2's
		 * warp instructions ran with fewer than 2 active lanes, almost all of them here): lanes reach a top-level leaf at different
		 * iterations, so running this ~100-instruction block whenever ANY lane wants it means running it for one lane.  Lanes
		 * therefore WAIT here until at least CRG_INST_MIN of them want an instance step, or no lane of the warp can take a node step. */
		{
			const bool wi = busy && tr.wants_instance();
			const unsigned mi = __ballot_sync(0xffffffffu, wi);
			if (mi) {
				bool go = __popc(mi) >= CRG_INST_MIN;
				if (!go) go = !__any_sync(0xffffffffu, busy && tr.wants_node());
				if (go && wi) { tr.instance_step(sc, &tc); ++steps; }
			}
		}
		/* Phase W: write back finished rays */
		if (busy && tr.done()) {
			wb.hit[ray] = make_float4(tr.best.t, tr.best.u, tr.best.v, __uint_as_float(tr.best.prim));
			wb.hitInst[ray] = tr.best.inst;
			unsigned key = 0u;                                   /* shading bucket for K4/K3 */
			if (tr.best.inst >= 0) {
				const DevInstance *inst = sc.instances + tr.best.inst;
				unsigned material;
				if (__ldg(&inst->kind) == CRS_INST_MESH) material = __ldg(&sc.spolys[__ldg(sc.slot_poly + tr.best.prim)].material);
				else material = __ldg(&inst->material);
				key = material + 1u < 255u ? material + 1u : 255u;
			}
			wb.hitKey[ray] = (unsigned char)key;
			atomicAdd(&s_hist[key], 1u);
			busy = false;
		} else if (busy && steps > CRG_MAX_STEPS) {              /* cannot happen for a finite BVH; never hang the GPU */
			atomicAdd(&wb.stats[7], 1ull);
			wb.hit[ray] = make_float4(CR_FLT_MAX, 0.f, 0.f, 0.f);
			wb.hitInst[ray] = -1;
			wb.hitKey[ray] = 0;
			atomicAdd(&s_hist[0], 1u);
			busy = false;
		}
	}
	__syncthreads();
	if (s_hist[threadIdx.x]) atomicAdd(&wb.hist[threadIdx.x], s_hist[threadIdx.x]);
	if (COUNT) {
		atomicAdd(&wb.stats[1], (unsigned long long)tc.pairs);
		atomicAdd(&wb.stats[2], (unsigned long long)tc.tris);
		atomicAdd(&wb.stats[3], (unsigned long long)tc.spheres);
		atomicAdd(&wb.stats[4], (unsigned long long)tc.insts);
	}
	if (blockIdx.x == 0 && threadIdx.x == 0) {
		atomicAdd(&wb.stats[0], (unsigned long long)n);          /* one ray per getClosestIsect (two streams may run two K2s) */
		wb.counts[cur ^ 1] = 0u;   /* K3 of this bounce appends survivors there */
	}
}

void crg_launch_generate(const DevScene &sc, const WaveBuffers &wb, const TileDesc &td, int grid, cudaStream_t st) {
	k_generate<<<grid, 256, 0, st>>>(sc, wb, td);
}
/* K2 is persistent: the grid is exactly the number of blocks the device can keep resident (3 per SM: the launch bounds
 * leave the compiler 80 registers per thread). */
#ifndef CRG_MAX_DEVICES
#define CRG_MAX_DEVICES 64
#endif
template <bool COUNT>
static void launch_trace_variant(const DevScene &sc, const WaveBuffers &wb, int cur, cudaStream_t st) {
	/* grid per DEVICE: the host mirror drives several GPUs from one process (one thread each), and the occupancy answer
	 * belongs to a device, not to the process */
	static int grids[CRG_MAX_DEVICES];
	static std::mutex grids_lock;
	int dev = 0;
	cudaGetDevice(&dev);
	int grid;
	{
		std::lock_guard<std::mutex> guard(grids_lock);
		int &g = grids[dev >= 0 && dev < CRG_MAX_DEVICES ? dev : 0];
		if (!g) {
			int sms = 0, occ = 0;
			cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
			cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_trace<COUNT>, 256, 0);
			g = sms * (occ > 0 ? occ : 1);
		}
		grid = g;
	}
	k_trace<COUNT><<<grid, 256, 0, st>>>(sc, wb, cur);
}

void crg_launch_trace(const DevScene &sc, const WaveBuffers &wb, int cur, bool count, cudaStream_t st) {
	if (count) launch_trace_variant<true>(sc, wb, cur, st);
	else launch_trace_variant<false>(sc, wb, cur, st);
}

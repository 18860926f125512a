/*
 * crgpu_shade.cu — K3 (shade + compaction), K5 (accumulate), sRGB8 conversion and the known-answer
 * kernel: see crgpu_wave.cuh.  The node interpreter and the fp64 libm stand-ins are real function
 * calls (__noinline__), so the scene descriptor is read through a pointer to its device copy.
 */
#include "crgpu_wave.cuh"
#include "crgpu_shade.cuh"

/* ---- K4: counting sort of the live rays by shading bucket --------------------------------------------------------------------
 * K2 left the bucket sizes in wb.hist[0..255].  Every block derives the same exclusive prefix, then ranks
 * its rays inside the block with shared-memory atomics and reserves one contiguous range per non-empty bucket
 * with ONE global atomicAdd (cursor = wb.hist[256+k]).  Output: perm[bucket_base + rank] = live index.
 * Order inside a bucket is arbitrary; results do not depend on it (every path carries its own RNG + id). */
#define CRG_BUCKET_ITEMS 8
__global__ void __launch_bounds__(256) k_bucket(WaveBuffers wb, int cur) {
	__shared__ unsigned s_base[256], s_cnt[256], s_off[256];
	const unsigned n = wb.counts[cur];
	const unsigned t = threadIdx.x;
	unsigned *__restrict__ sizes = wb.hist;
	unsigned *__restrict__ cursors = wb.hist + 256;
	const unsigned char *__restrict__ keys = wb.hitKey;
	unsigned *__restrict__ out = wb.perm;
	s_cnt[t] = sizes[t];
	__syncthreads();
	if (t == 0u) { unsigned acc = 0u; for (int k = 0; k < 256; ++k) { s_base[k] = acc; acc += s_cnt[k]; } }
	__syncthreads();
	if (blockIdx.x == 0u && t == 0u) wb.counts[4] = s_base[1];      /* = bucket 0's size: perm[0 .. counts[4]) are the misses (K3 split) */
	const unsigned chunk = 256u * CRG_BUCKET_ITEMS;
	for (unsigned c0 = blockIdx.x * chunk; c0 < n; c0 += gridDim.x * chunk) {
		s_cnt[t] = 0u;
		__syncthreads();
		unsigned key[CRG_BUCKET_ITEMS], rank[CRG_BUCKET_ITEMS];
#pragma unroll
		for (int k = 0; k < CRG_BUCKET_ITEMS; ++k) {
			const unsigned i = c0 + (unsigned)k * 256u + t;
			key[k] = 0xffffffffu;
			if (i < n) { key[k] = keys[i]; rank[k] = atomicAdd(&s_cnt[key[k]], 1u); }
		}
		__syncthreads();
		s_off[t] = s_cnt[t] ? atomicAdd(&cursors[t], s_cnt[t]) : 0u;
		__syncthreads();
#pragma unroll
		for (int k = 0; k < CRG_BUCKET_ITEMS; ++k) {
			const unsigned i = c0 + (unsigned)k * 256u + t;
			if (key[k] != 0xffffffffu) out[s_base[key[k]] + s_off[key[k]] + rank[k]] = i;
		}
		__syncthreads();
	}
}

/* ---- one bounce of pathTrace's loop body for one path (pathtrace.c:38-57), shared by K3 and the tail kernel -----------------
 * Radiance goes to L[path id].  The reference accumulates into finalColor = (0,0,0) (pathtrace.c:34); the first
 * contribution is therefore written as 0.0f + x (bit-identical, also for x = -0) WITHOUT reading L, and the top bit
 * of the carried id remembers that L holds a value; a path that ends without any contribution writes zeros.  So K1
 * never has to clear L and most paths touch their L record exactly once. */
#define CRG_ID_HAS_L 0x80000000u

CRD void cr_add_radiance(float4 *__restrict__ Lbuf, unsigned &id, float r, float g, float b) {
	const unsigned slot = id & ~CRG_ID_HAS_L;
	float4 L = (id & CRG_ID_HAS_L) ? Lbuf[slot] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
	L.x = L.x + r; L.y = L.y + g; L.z = L.z + b;
	Lbuf[slot] = L;
	id |= CRG_ID_HAS_L;
}
CRD void cr_finish_path(float4 *__restrict__ Lbuf, unsigned id) {
	if (!(id & CRG_ID_HAS_L)) Lbuf[id] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}

/* returns true when the path continues with (p_next, d_next) and the updated weight / rng / id */
template <bool X, bool MAYBE_MISS = true>
CRD bool cr_shade_one(const DevScene &sc, float4 *__restrict__ Lbuf, v3 o, v3 d, const Hit &hit, float &wr, float &wg, float &wbl,
					  unsigned &id, uint64_t &rng, int depth, int maxDepth, v3 &p_next, v3 &d_next) {
	if (MAYBE_MISS && hit.inst < 0) {                                                               /* pathtrace.c:39-42 */
		const col4 bg = cr_sample_background<X>(sc, d);
		cr_add_radiance(Lbuf, id, wr * bg.r, wg * bg.g, wbl * bg.b);
		return false;
	}
	Rec rec;
	const int material = cr_reconstruct_hit(sc, o, d, hit, rec, false);
	const DevMaterial mat = sc.materials[material];
	if (mat.flags & 2u)                                                               /* pathtrace.c:44 (x + w*0 == x) */
		cr_add_radiance(Lbuf, id, wr * mat.emission[0], wg * mat.emission[1], wbl * mat.emission[2]);
	if (depth + 1 < maxDepth) {                                                       /* else: the loop ends, the sample is unused */
		const BsdfSample s = cr_sample_bsdf<X>(sc, mat.bsdf, rng, rec);              /* pathtrace.c:46-48 */
		float probability = 1.0f;
		bool cont = true;
		if (depth >= 4) {                                                             /* pathtrace.c:50-55 */
			probability = CR_MAX(s.color.r, CR_MAX(s.color.g, s.color.b));
			if (cr_draw(rng) > probability) cont = false;
		}
		if (cont) {
			const float inv = cr_div(1.0f, probability);                              /* pathtrace.c:57 */
			wr = (s.color.r * wr) * inv; wg = (s.color.g * wg) * inv; wbl = (s.color.b * wbl) * inv;
			p_next = rec.p; d_next = s.out;
			return true;
		}
	}
	cr_finish_path(Lbuf, id);
	return false;
}

/* ---- K3 (+ compaction) ----------------------------------------------------------------------------------------------
 * Two launches over the bucket order: PART 1 = the misses (bucket 0 = perm[0 .. counts[4]): background lookup + radiance, the
 * path always ends, nothing to compact), 4 blocks per SM; PART 2 = the hits (perm[counts[4] .. n)), 3 blocks per SM.  The miss
 * half needs a third of the registers of the hit half, so it runs at higher occupancy; on hdr.json 40% of all rays are misses. */
template <int PART, bool X>
__global__ void __launch_bounds__(256, PART == 1 ? 4 : 3) k_shade(const DevScene *__restrict__ scp, WaveBuffers wb, int cur, int depth, int maxDepth) {
	const DevScene &sc = *scp;
	const unsigned n = wb.counts[cur];
	const int nxt = cur ^ 1;
	const unsigned stride = gridDim.x * blockDim.x;
	if (PART == 1) {
		const unsigned n0 = wb.counts[4];
		for (unsigned j = blockIdx.x * blockDim.x + threadIdx.x; j < n0; j += stride) {
			const unsigned i = wb.perm[j];
			const float4 a = wb.stA[cur][i];
			const float4 b = wb.stB[cur][i];
			const uint4 c = wb.stC[cur][i];
			unsigned id = c.y;
			const col4 bg = cr_sample_background<X>(sc, v3make(a.w, b.x, b.y));                 /* pathtrace.c:39-42 */
			cr_add_radiance(wb.L, id, b.z * bg.r, b.w * bg.g, __uint_as_float(c.x) * bg.b);
		}
		return;
	}
	if (blockIdx.x == 0 && threadIdx.x == 0) wb.counts[2] = 0u;   /* K2's work counter, for the next bounce */
	if (blockIdx.x == 0) { wb.hist[threadIdx.x] = 0u; wb.hist[256 + threadIdx.x] = 0u; }   /* K2/K4 histogram + cursors (blockDim.x == 256) */
	const unsigned lane = threadIdx.x & 31u;
	/* whole warps iterate together so the ballot below is convergent */
	const unsigned first = wb.counts[4];
	const unsigned nround = first + ((n - first + 31u) & ~31u);
	for (unsigned j = first + blockIdx.x * blockDim.x + threadIdx.x; j < nround; j += stride) {
		bool alive = false;
		v3 p_next = v3make(0, 0, 0), d_next = v3make(0, 0, 0);
		float wr = 0.f, wg = 0.f, wbl = 0.f;
		unsigned id = 0u;
		uint64_t rng = 0ull;
		if (j < n) {
			const unsigned i = wb.perm[j];     /* bucket order: a warp shades one material */
			const float4 a = wb.stA[cur][i];
			const float4 b = wb.stB[cur][i];
			const uint4 c = wb.stC[cur][i];
			const float4 hq = wb.hit[i];
			Hit hit;
			hit.t = hq.x; hit.u = hq.y; hit.v = hq.z; hit.prim = __float_as_uint(hq.w);
			hit.inst = wb.hitInst[i];
			wr = b.z; wg = b.w; wbl = __uint_as_float(c.x);
			id = c.y;
			rng = (uint64_t)c.z | ((uint64_t)c.w << 32);
			alive = cr_shade_one<X, false>(sc, wb.L, v3make(a.x, a.y, a.z), v3make(a.w, b.x, b.y), hit, wr, wg, wbl, id, rng, depth, maxDepth, p_next, d_next);
		}
		/* order-preserving warp compaction, one atomic per warp */
		const unsigned mask = __ballot_sync(0xffffffffu, alive);
		if (mask) {
			unsigned base = 0u;
			if (lane == 0u) base = atomicAdd(&wb.counts[nxt], (unsigned)__popc(mask));
			base = __shfl_sync(0xffffffffu, base, 0);
			if (alive) {
				const unsigned k = base + (unsigned)__popc(mask & ((1u << lane) - 1u));
				wb.stA[nxt][k] = make_float4(p_next.x, p_next.y, p_next.z, d_next.x);
				wb.stB[nxt][k] = make_float4(d_next.y, d_next.z, wr, wg);
				wb.stC[nxt][k] = make_uint4(__float_as_uint(wbl), id, (unsigned)(rng & 0xffffffffull), (unsigned)(rng >> 32));
			}
		}
	}
}

/* ---- tail kernel: when only a handful of paths is left, finish them in ONE launch -------------------------------------------
 * Late bounces hold few rays (hdr.json: <0.1% of the batch after 10 bounces; refraction.json keeps a trickle alive for
 * hundreds of bounces), but every bounce still costs three launches and lasts as long as its slowest ray (~0.2 ms).
 * From bounce CRG_TAIL_FROM on, this kernel is launched before K2: if at most CRG_TAIL_MAX rays are left it runs each
 * remaining path to completion (trace + shade in a per-thread loop — the same device functions, the same draws) and
 * zeroes the live count, so the K2/K4/K3 launches that follow find nothing to do. */
#define CRG_TAIL_MAX 16384u

template <bool X>
__global__ void __launch_bounds__(128) k_tail(const DevScene *__restrict__ scp, WaveBuffers wb, int cur, int depth0, int maxDepth) {
	const DevScene &sc = *scp;
	const unsigned n = wb.counts[cur];
	if (n == 0u || n > CRG_TAIL_MAX) return;
	for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const float4 a = wb.stA[cur][i];
		const float4 b = wb.stB[cur][i];
		const uint4 c = wb.stC[cur][i];
		v3 o = v3make(a.x, a.y, a.z), d = v3make(a.w, b.x, b.y);
		float wr = b.z, wg = b.w, wbl = __uint_as_float(c.x);
		unsigned id = c.y;
		uint64_t rng = (uint64_t)c.z | ((uint64_t)c.w << 32);
		unsigned long long rays = 0ull;
		for (int depth = depth0; depth < maxDepth; ++depth) {
			const Hit hit = cr_closest_hit<false>(sc, o, d, nullptr);
			++rays;
			v3 p_next, d_next;
			if (!cr_shade_one<X>(sc, wb.L, o, d, hit, wr, wg, wbl, id, rng, depth, maxDepth, p_next, d_next)) break;
			o = p_next; d = d_next;
		}
		atomicAdd(&wb.stats[0], rays);
	}
	/* the last block to finish clears the queue (every block has read n by then) */
	__shared__ unsigned s_last;
	__syncthreads();
	if (threadIdx.x == 0) { __threadfence(); s_last = atomicAdd(&wb.counts[3], 1u) == gridDim.x - 1u; }
	__syncthreads();
	if (s_last && threadIdx.x == 0) { wb.counts[cur] = 0u; wb.counts[cur ^ 1] = 0u; wb.counts[3] = 0u; }
}

/* ---- K5 ------------------------------------------------------------------------------------------------------------------ */
__global__ void __launch_bounds__(256) k_accumulate(float *__restrict__ fb, const float4 *__restrict__ L, TileDesc td,
													 int image_width, int image_height) {
	const unsigned tile_pixels = td.npix;
	for (unsigned px = blockIdx.x * blockDim.x + threadIdx.x; px < tile_pixels; px += gridDim.x * blockDim.x) {
		int x, y;
		crg_pixel_xy(td, px, x, y);
		float *dst = fb + ((size_t)x + (size_t)(image_height - (y + 1)) * (size_t)image_width) * 3u;  /* texture.c:24-28 */
		float r = dst[0], g = dst[1], b = dst[2];
		for (int pl = 0; pl < td.pass_count; ++pl) {
			const float4 s = L[(size_t)pl * tile_pixels + px];
			const int completed = td.pass_begin + pl + 1;                                     /* renderer.c:288-291 */
			const float k = (float)(completed - 1);
			const float t = cr_div(1.0f, (float)completed);
			r = (r * k + s.x) * t; g = (g * k + s.y) * t; b = (b * k + s.z) * t;
		}
		dst[0] = r; dst[1] = g; dst[2] = b;
	}
}

/* colorToSRGB + setPixel(char_p): renderer.c:297-300, texture.c:19-21 */
__global__ void k_to_srgb8(const float *__restrict__ fb, uint8_t *__restrict__ out, size_t n) {
	for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
		const float c = cr_linear_to_srgb(fb[i]);
		const float s = CR_MIN(c * 255.0f, 255.0f);
		/* (unsigned char) of a negative/NaN float is UB in C; x86 cvttss2si + truncation gives the low byte */
		out[i] = (uint8_t)(cr_f2i(s) & 0xff);
	}
}

/* ---- known-answer kernel (parity tests): one thread per (x, y, pass) ---------------------------------------------------------- */
struct HitKat {
	int32_t x, y, pixIdx, instIndex, polyIndex;
	float o[3], d[3];
	float distance, uv[2];
	float hitPoint[3], normal[3];
	float emission[3];
	float out[3], color[4];
	float nextDraw;
	float pad[9];
};

__global__ void k_kat(const DevScene *__restrict__ scp, const int32_t *__restrict__ xyp, int count, HitKat *__restrict__ outv) {
	const DevScene &sc = *scp;
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= count) return;
	HitKat k;
	memset(&k, 0, sizeof k);
	const int x = xyp[3 * i], y = xyp[3 * i + 1], pass = xyp[3 * i + 2];
	k.x = x; k.y = y; k.pixIdx = y * (int)sc.image_width + x;
	uint64_t rng = cr_rng_init((uint32_t)k.pixIdx, (uint32_t)pass, sc.sample_count);
	v3 o, d;
	cr_camera_ray(sc.cam, x, y, rng, o, d);
	k.o[0] = o.x; k.o[1] = o.y; k.o[2] = o.z; k.d[0] = d.x; k.d[1] = d.y; k.d[2] = d.z;
	const Hit hit = cr_closest_hit<false>(sc, o, d, nullptr);
	k.instIndex = hit.inst;
	BsdfSample s;
	if (hit.inst < 0) {
		k.polyIndex = -1;
		s.out = v3make(0.f, 0.f, 0.f);
		s.color = cr_sample_background<true>(sc, d);
	} else {
		Rec rec;
		const int material = cr_reconstruct_hit(sc, o, d, hit, rec, true);
		const DevInstance *inst = sc.instances + hit.inst;
		k.polyIndex = inst->kind == CRS_INST_MESH ? (int)sc.slot_poly[hit.prim] : -1;
		k.distance = hit.t; k.uv[0] = rec.uv.x; k.uv[1] = rec.uv.y;
		k.hitPoint[0] = rec.p.x; k.hitPoint[1] = rec.p.y; k.hitPoint[2] = rec.p.z;
		k.normal[0] = rec.n.x; k.normal[1] = rec.n.y; k.normal[2] = rec.n.z;
		const DevMaterial mat = sc.materials[material];
		k.emission[0] = mat.emission[0]; k.emission[1] = mat.emission[1]; k.emission[2] = mat.emission[2];
		s = cr_sample_bsdf<true>(sc, mat.bsdf, rng, rec);
	}
	k.out[0] = s.out.x; k.out[1] = s.out.y; k.out[2] = s.out.z;
	k.color[0] = s.color.r; k.color[1] = s.color.g; k.color[2] = s.color.b; k.color[3] = s.color.a;
	k.nextDraw = cr_draw(rng);
	outv[i] = k;
}

void crg_launch_bucket(const WaveBuffers &wb, int cur, int grid, cudaStream_t st) {
	k_bucket<<<grid, 256, 0, st>>>(wb, cur);
}
/* X (the last template argument): the scene contains node kinds only the complete interpreter knows (DevScene::has_xnodes, set at
 * upload) — every other scene runs the kernels in which that interpreter is not even linked */
void crg_launch_tail(const DevScene *dsc, const WaveBuffers &wb, int cur, int depth, int maxDepth, bool xnodes, cudaStream_t st) {
	if (xnodes) k_tail<true><<<128, 128, 0, st>>>(dsc, wb, cur, depth, maxDepth);
	else k_tail<false><<<128, 128, 0, st>>>(dsc, wb, cur, depth, maxDepth);
}
void crg_launch_shade(const DevScene *dsc, const WaveBuffers &wb, int cur, int depth, int maxDepth, bool xnodes, int grid, cudaStream_t st) {
	if (xnodes) {
		k_shade<1, true><<<grid, 256, 0, st>>>(dsc, wb, cur, depth, maxDepth);
		k_shade<2, true><<<grid, 256, 0, st>>>(dsc, wb, cur, depth, maxDepth);
	} else {
		k_shade<1, false><<<grid, 256, 0, st>>>(dsc, wb, cur, depth, maxDepth);
		k_shade<2, false><<<grid, 256, 0, st>>>(dsc, wb, cur, depth, maxDepth);
	}
}
void crg_launch_accumulate(float *fb, const float4 *L, const TileDesc &td, int W, int H, int grid, cudaStream_t st) {
	k_accumulate<<<grid, 256, 0, st>>>(fb, L, td, W, H);
}
void crg_launch_to_srgb8(const float *fb, uint8_t *out, size_t n, int grid, cudaStream_t st) {
	k_to_srgb8<<<grid, 256, 0, st>>>(fb, out, n);
}
void crg_launch_kat(const DevScene *dsc, const int32_t *xyp, int count, void *out, cudaStream_t st) {
	k_kat<<<(count + 63) / 64, 64, 0, st>>>(dsc, xyp, count, static_cast<HitKat *>(out));
}
static_assert(sizeof(HitKat) == 160, "HitKat must match struct hit_kat of oracle/ref_harness.c");

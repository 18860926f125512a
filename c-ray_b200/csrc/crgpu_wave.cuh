/*
 * crgpu_wave.cuh — wavefront buffers and kernel launchers shared by the translation units of libcrgpu.so.
 *
 * One `crgpu_render_tile` call processes a tile rectangle in batches of B passes; a batch has
 * N = tile_pixels * B paths, path id = p_local * tile_pixels + pixel_local.  Per batch:
 *
 *   K1 k_generate    initSampler + getCameraRay for every path            (sampler.c:41-44, camera.c:58-87)
 *   per bounce:
 *   K2 k_trace       closest hit of every live ray                        (pathtrace.c:38 → bvh.c, poly.c, sphere.c)
 *   K4 k_bucket      counting sort of the live rays by shading bucket (miss / material id) so that the
 *                    32 lanes of a K3 warp run the same node graph (K2 fills the histogram)
 *   K3 k_shade       miss → background, hit → emission, bsdf sample, Russian roulette, weight update;
 *                    survivors are COMPACTED into the other half of the ping-pong ray buffers with one
 *                    warp-ballot + one atomicAdd per warp (K4 is fused into K3)   (pathtrace.c:39-57)
 *   K5 k_accumulate  running average of the B pass samples into the fp32 framebuffer, in pass order
 *                                                                         (renderer.c:288-294)
 *
 * Path state in HBM (SoA of 16-byte vectors, always read/written at the COMPACT live index, so every
 * access is a coalesced 128-bit transaction):
 *   stA = (o.x, o.y, o.z, d.x)   stB = (d.y, d.z, weight.r, weight.g)   stC = (weight.b, path id, rng lo, rng hi)
 *   hit = (t, u, v, prim slot)   hitInst = instance index or -1
 *   L[path id] = (r, g, b, -)    radiance of the path, written at termination / emissive hits
 * The queue order never affects results: every path carries its own RNG state and id.
 */
#pragma once
#include <cuda_runtime.h>
#include "crgpu_scene.cuh"

struct WaveBuffers {
	float4 *stA[2];
	float4 *stB[2];
	uint4  *stC[2];
	float4 *hit;
	int    *hitInst;
	float4 *L;
	unsigned char *hitKey;  /* shading bucket of the hit: 0 = miss, else min(material+1, 255) */
	unsigned *perm;         /* K4 output: live indices grouped by bucket */
	unsigned *hist;         /* [256] bucket sizes (filled by K2), [256..511] K4 cursors */
	unsigned *counts;       /* [0],[1]: live counts of the ping-pong halves; [2]: K2's work counter (next ray to hand out); [3]: tail-kernel block counter; [4]: number of misses of this bounce (K4 -> K3 split) */
	unsigned long long *stats; /* [0] rays, [1] pairs, [2] tris, [3] spheres, [4] insts */
};

struct TileDesc {
	int x0, y0, tw, th;     /* tile origin and size (pixels); y up */
	int pass_begin, pass_count; /* this batch */
	const uint32_t *pixels; /* NULL: the pixel set is the rectangle above; else an explicit list x | y << 16 (a union of tiles) */
	unsigned npix;          /* number of pixels in the set */
};

__device__ __forceinline__ void crg_pixel_xy(const TileDesc &td, unsigned px, int &x, int &y) {
	if (td.pixels) { const uint32_t p = __ldg(td.pixels + px); x = (int)(p & 0xffffu); y = (int)(p >> 16); }
	else { x = td.x0 + (int)(px % (unsigned)td.tw); y = td.y0 + (int)(px / (unsigned)td.tw); }
}

/* launchers (defined in crgpu_trace.cu / crgpu_shade.cu); `dsc` is the device copy of `sc` */
void crg_launch_pixel_list(uint32_t *pixels, const int4 *rects, const unsigned *offs, int nrects, cudaStream_t st);
void crg_launch_generate(const DevScene &sc, const WaveBuffers &wb, const TileDesc &td, int grid, cudaStream_t st);
void crg_launch_trace(const DevScene &sc, const WaveBuffers &wb, int cur, bool count, cudaStream_t st);
void crg_launch_bucket(const WaveBuffers &wb, int cur, int grid, cudaStream_t st);
void crg_launch_tail(const DevScene *dsc, const WaveBuffers &wb, int cur, int depth, int maxDepth, bool xnodes, cudaStream_t st);
void crg_launch_shade(const DevScene *dsc, const WaveBuffers &wb, int cur, int depth, int maxDepth, bool xnodes, int grid, cudaStream_t st);
void crg_launch_accumulate(float *fb, const float4 *L, const TileDesc &td, int W, int H, int grid, cudaStream_t st);
void crg_launch_to_srgb8(const float *fb, uint8_t *out, size_t n, int grid, cudaStream_t st);
void crg_launch_kat(const DevScene *dsc, const int32_t *xyp, int count, void *out, cudaStream_t st);

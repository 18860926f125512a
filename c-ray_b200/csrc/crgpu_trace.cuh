/*
 * crgpu_trace.cuh — camera ray generation and two-level BVH closest-hit query (device functions).
 *
 * Restates, over the device layout of crgpu_scene.cuh:
 *   getCameraRay            reference src/datatypes/camera.c:50-87
 *   traverseBvhGeneric      reference src/accelerators/bvh.c:354-441 (+ intersectNode :326-352)
 *   intersectTopLevelLeaf   bvh.c:468-486      intersectBottomLevelLeaf  bvh.c:443-462
 *   intersectSphere/Mesh    src/datatypes/instance.c:45-60, 169-185 (closest-hit part)
 *   rayIntersectsWithPolygon src/datatypes/poly.c:17-53      intersect  src/datatypes/sphere.c:20-50
 *
 * The traversal visits nodes and primitives in EXACTLY the reference order (nearer child first,
 * farther pushed; both children tested with the maxDist valid before either leaf is processed), so
 * the closest hit — including exact-tie winners — is the reference's.
 */
#pragma once
#include "crgpu_math.cuh"
#include "crgpu_scene.cuh"

struct Hit {
	float t, u, v;
	int   inst;          /* -1 = miss */
	uint32_t prim;       /* global prim slot of the winning triangle */
};

struct TraceCounters { unsigned pairs, tris, spheres, insts; };

/* ---- camera.c:50-87 ---------------------------------------------------------------------------------------- */
CRD float cr_triangle_distribution(float v) {
	const float orig = v * 2.0f - 1.0f;
	v = cr_div(orig, cr_sqrtf(fabsf(orig)));
	v = cr_clamp(v, -1.0f, 1.0f);
	v = v - ((orig >= 0.0f) ? 1.0f : -1.0f);
	return v;
}

CRD void cr_camera_ray(const DevCamera &cam, int x, int y, uint64_t &rng, v3 &o, v3 &d) {
	const v3 right = v3make(cam.right[0], cam.right[1], cam.right[2]);
	const v3 up = v3make(cam.up[0], cam.up[1], cam.up[2]);
	const v3 forward = v3make(cam.forward[0], cam.forward[1], cam.forward[2]);
	const float jitterX = cr_triangle_distribution(cr_draw(rng));
	const float jitterY = cr_triangle_distribution(cr_draw(rng));
	const v3 pixX = v3scale(right, cr_div(cam.sensor_x, (float)cam.width));
	const v3 pixY = v3scale(up, cr_div(cam.sensor_y, (float)cam.height));
	const v3 pixV = v3add(forward, v3add(v3scale(pixX, (float)x - (float)cam.width * 0.5f + jitterX + 0.5f),
										 v3scale(pixY, (float)y - (float)cam.height * 0.5f + jitterY + 0.5f)));
	o = v3make(0.0f, 0.0f, 0.0f);
	d = v3norm(pixV);
	if (cam.aperture > 0.0f) {
		const float ft = cr_div(cam.focal_distance, v3dot(d, forward));
		const v3 focus = v3add(o, v3scale(d, ft));
		const float rr = cr_sqrtf(cr_draw(rng));                               /* vector.h:194-198 */
		const float theta = (cr_draw(rng) * (2.0f * CR_PI - 0.0f)) + 0.0f;
		float sn, cs;
		cr_sincosf(theta, &sn, &cs);
		const float lx = (rr * cs) * cam.aperture, ly = (rr * sn) * cam.aperture;
		o = v3add(o, v3add(v3scale(right, lx), v3scale(up, ly)));
		d = v3norm(v3sub(focus, o));
	}
	o = xf_point(cam.A, o);
	d = xf_vector(cam.A, d);
}

/* ---- bvh.c:326-352 -------------------------------------------------------------------------------------------- */
struct RaySetup {
	v3 invDir, scaledStart;
	bool ox, oy, oz;
	unsigned deg;      /* bit a set: 1/d[a] is +-inf (d[a] is +-0 or denormal) — see cr_node_test */
};

CRD RaySetup cr_ray_setup(v3 o, v3 d) {                                                /* bvh.c:369-376 */
	RaySetup s;
	s.ox = (__float_as_uint(d.x) >> 31) != 0u;
	s.oy = (__float_as_uint(d.y) >> 31) != 0u;
	s.oz = (__float_as_uint(d.z) >> 31) != 0u;
	s.invDir = v3make(cr_div(1.0f, d.x), cr_div(1.0f, d.y), cr_div(1.0f, d.z));
	s.scaledStart = v3scale(v3mul(o, s.invDir), -1.0f);
	s.deg = (isinf(s.invDir.x) ? 1u : 0u) | (isinf(s.invDir.y) ? 2u : 0u) | (isinf(s.invDir.z) ? 4u : 0u);
	return s;
}

/* bvh.c:318-324: `fastMultiplyAdd` is fmaf() when the compiler defines FP_FAST_FMAF (the reference's stock
 * -march=native build) and a*b+c otherwise (the strict oracle build).  The slab test only decides which nodes
 * are ENTERED, never a hit distance, and both variants are conservative; the survey measured bit-identical
 * framebuffers between them on hdr.json and venus.json, and tests/test_gpu_parity.py holds the fused variant to
 * exact hit records against the un-fused oracle.  Fused = 6 FFMA per child instead of 6 FMUL + 6 FADD. */
#define CR_SLAB_MAD(a, b, c) __fmaf_rn((a), (b), (c))

/* Slab test of one child.  For ordinary rays this is intersectNode verbatim (bvh.c:326-352).
 *
 * Degenerate axes.  When a direction component is exactly 0 the reference computes b*inf + (-o*inf),
 * which is NaN for most bounds; its NaN-tolerant min/max chain then silently DROPS that axis (and, by
 * propagation, the x or y axis before it), so such a ray "enters" a large part of the BVH — up to
 * ~115,000 of Venus' 229,087 nodes per ray (measured with the oracle on hdr.json, horizon rays with
 * d.y == 0).  That is harmless on a CPU (~1 ms) but one GPU thread would need ~50-150 ms while the
 * whole wavefront waits.  The reference's degenerate test is a pure superset of the exact slab test and
 * the Möller–Trumbore test decides every hit on its own, so culling with the exact test (axis with
 * d == 0: inside the slab iff lo <= o <= hi) returns the same closest hit; the two could only differ
 * for a ray that grazes a triangle within one ulp of its leaf's bounding box, on an already
 * measure-zero ray (~1e-13 per ray).  Rays without a zero component take the verbatim path. */
CRD bool cr_node_test(const float *b, const RaySetup &r, v3 o, float maxDist, float &tEntry) {
	float tMinX = CR_SLAB_MAD((r.ox ? b[1] : b[0]), r.invDir.x, r.scaledStart.x);
	float tMaxX = CR_SLAB_MAD((r.ox ? b[0] : b[1]), r.invDir.x, r.scaledStart.x);
	float tMinY = CR_SLAB_MAD((r.oy ? b[3] : b[2]), r.invDir.y, r.scaledStart.y);
	float tMaxY = CR_SLAB_MAD((r.oy ? b[2] : b[3]), r.invDir.y, r.scaledStart.y);
	float tMinZ = CR_SLAB_MAD((r.oz ? b[5] : b[4]), r.invDir.z, r.scaledStart.z);
	float tMaxZ = CR_SLAB_MAD((r.oz ? b[4] : b[5]), r.invDir.z, r.scaledStart.z);
	if (r.deg) {
		const float inf = __int_as_float(0x7f800000);
		if (r.deg & 1u) { const bool in = (b[0] <= o.x) && (o.x <= b[1]); tMinX = in ? -inf : inf; tMaxX = in ? inf : -inf; }
		if (r.deg & 2u) { const bool in = (b[2] <= o.y) && (o.y <= b[3]); tMinY = in ? -inf : inf; tMaxY = in ? inf : -inf; }
		if (r.deg & 4u) { const bool in = (b[4] <= o.z) && (o.z <= b[5]); tMinZ = in ? -inf : inf; tMaxZ = in ? inf : -inf; }
	}
	float tMin = tMinX > tMinY ? tMinX : tMinY;
	float tMax = tMaxX < tMaxY ? tMaxX : tMaxY;
	tMin = tMin > tMinZ ? tMin : tMinZ;
	tMax = tMax < tMaxZ ? tMax : tMaxZ;
	tMin = tMin > 0 ? tMin : 0;
	tMax = tMax < maxDist ? tMax : maxDist;
	tEntry = tMin;
	return tMin <= tMax;
}

/* rayIntersectsWithPolygon over one leaf (bvh.c:443-462 + poly.c:17-53); tris already offset to the BVH's first slot */
template <bool COUNT>
CRD bool cr_leaf_tris(const PackedTri *__restrict__ tris, uint32_t slot_base, uint32_t first, uint32_t count,
					  v3 o, v3 d, Hit &best, TraceCounters *ctr) {
	bool found = false;
	for (uint32_t i = 0; i < count; ++i) {
		const float4 *t4 = reinterpret_cast<const float4 *>(tris + first + i);
		const float4 a = __ldg(t4 + 0), b = __ldg(t4 + 1), c4 = __ldg(t4 + 2);
		if (COUNT) ctr->tris++;
		const v3 v0 = v3make(a.x, a.y, a.z), e1 = v3make(a.w, b.x, b.y), e2 = v3make(b.z, b.w, c4.x);
		const v3 n = v3make(c4.y, c4.z, c4.w);
		const v3 c = v3sub(v0, o);
		const v3 r = v3cross(d, c);
		const float invDet = cr_div(1.0f, v3dot(n, d));
		const float u = v3dot(r, e2) * invDet;
		const float v = v3dot(r, e1) * invDet;
		if (u >= 0.0f && v >= 0.0f && u + v <= 1.0f) {
			const float t = v3dot(n, c) * invDet;
			if (t >= 0.0f && t < best.t) {
				best.t = t; best.u = u; best.v = v;
				best.prim = slot_base + first + i;
				found = true;
			}
		}
	}
	return found;
}

/* two leaves back to back: slots [firstA, firstA+nA) then [firstB, firstB+nB) */
template <bool COUNT>
CRD bool cr_leaf_tris2(const PackedTri *__restrict__ tris, uint32_t slot_base, uint32_t firstA, uint32_t nA, uint32_t firstB, uint32_t nB,
					   v3 o, v3 d, Hit &best, TraceCounters *ctr) {
	bool found = false;
	const uint32_t total = nA + nB;
	for (uint32_t k = 0; k < total; ++k) {
		const uint32_t slot = k < nA ? firstA + k : firstB + (k - nA);
		const float4 *t4 = reinterpret_cast<const float4 *>(tris + slot);
		const float4 a = __ldg(t4 + 0), b = __ldg(t4 + 1), c4 = __ldg(t4 + 2);
		if (COUNT) ctr->tris++;
		const v3 v0 = v3make(a.x, a.y, a.z), e1 = v3make(a.w, b.x, b.y), e2 = v3make(b.z, b.w, c4.x);
		const v3 n = v3make(c4.y, c4.z, c4.w);
		const v3 c = v3sub(v0, o);
		const v3 r = v3cross(d, c);
		const float invDet = cr_div(1.0f, v3dot(n, d));
		const float u = v3dot(r, e2) * invDet;
		const float v = v3dot(r, e1) * invDet;
		if (u >= 0.0f && v >= 0.0f && u + v <= 1.0f) {
			const float t = v3dot(n, c) * invDet;
			if (t >= 0.0f && t < best.t) {
				best.t = t; best.u = u; best.v = v;
				best.prim = slot_base + slot;
				found = true;
			}
		}
	}
	return found;
}

CRD bool cr_sphere_test(v3 o, v3 d, float radius, float &dist) {                   /* sphere.c:20-50 */
	const float A = v3dot(d, d);
	const float B = 2.0f * v3dot(d, o);
	const float C = v3dot(o, o) - (radius * radius);
	const float disc = B * B - 4.0f * A * C;
	if (disc < 0.0f) return false;
	const float sq = cr_sqrtf(disc);
	float t0 = cr_div(-B + sq, 2.0f);
	const float t1 = cr_div(-B - sq, 2.0f);
	if (t0 > t1 && t1 > 0.0f) t0 = t1;
	if (t0 < 0.00001f || t0 > dist) return false;
	dist = t0;
	return true;
}

/* object-space ray of an instance: transformRay(Ainv) + rayOffset advance (instance.c:47-50, 170-174) */
CRD void cr_object_ray(const float *Ainv, float ray_offset, v3 o, v3 d, v3 &oo, v3 &od) {
	oo = xf_point(Ainv, o);
	od = xf_vector(Ainv, d);
	oo = v3add(oo, v3scale(od, ray_offset));
}

#define CRG_END 0xffffffffu

/* getClosestIsect (pathtrace.c:26-30) = traverseTopLevelBvh → intersectTopLevelLeaf → intersectMesh →
 * traverseBottomLevelBvh, flattened into ONE loop so that the 32 lanes of a warp stay convergent:
 * every iteration a lane performs either one child-pair step (top OR bottom level — same code, only
 * the base pointer and the ray registers differ) or one instance step (transform the ray into the
 * next instance of a pending top-level leaf; spheres are tested on the spot, meshes switch the lane
 * to the bottom level).  The reference's recursion (a whole bottom-level traversal nested inside a
 * top-level leaf loop) serialised divergent lanes: ncu measured 3-6 active threads per warp.
 *
 * Order of evaluation is the reference's: both children are tested against the closest distance known
 * BEFORE either leaf is processed; left leaf, then right leaf; nearer internal child next, farther one
 * pushed; instances of a leaf in primIndices order; strict t < distance for triangles, t <= distance
 * for spheres.  The reference's `maxDist` copies always equal isect->distance at the time of a node
 * test (they are refreshed after every leaf that found something), so best.t is used directly. */
template <bool COUNT>
struct Traversal {
	Hit best;
	v3 wo, wd;             /* world ray */
	v3 o, d;               /* ray of the current level */
	RaySetup rs;
	const PairNode *__restrict__ base;
	const PackedTri *__restrict__ tris;
	uint32_t slotBase, node, topNext;
	uint32_t pendA, cntA, pendB, cntB;     /* pending top-level leaf items: A (left leaf) before B (right leaf) */
	int sp, spBase, curInst;
	bool bottom, instHit;
	uint32_t *stack;       /* 2*CRG_MAX_STACK+2 entries of thread-local memory, owned by the caller (keeps the scalars in registers) */

	CRD bool done() const { return !bottom && (cntA | cntB) == 0u && node == CRG_END; }

	CRD void begin(const DevScene &sc, v3 ro, v3 rd) {
		best.t = CR_FLT_MAX; best.u = 0.0f; best.v = 0.0f; best.inst = -1; best.prim = 0u;
		wo = ro; wd = rd; o = ro; d = rd;
		rs = cr_ray_setup(o, d);
		base = sc.pairs + sc.top.pair_offset;
		tris = sc.tris;
		slotBase = 0u; node = 0u; topNext = CRG_END;
		pendA = 0u; cntA = 0u; pendB = 0u; cntB = 0u;
		sp = 0; spBase = 0; curInst = -1;
		bottom = false; instHit = false;
		if (sc.top.node_count < 1) {                                               /* bvh.c:362-365 */
			node = CRG_END;
		} else if (sc.top.node_count == 1) {                                       /* bvh.c:382-387 */
			float te;
			node = CRG_END;
			if (cr_node_test(sc.top.root_bounds, rs, o, best.t, te)) { pendA = sc.top.root_first; cntA = sc.top.root_count; }
		}
	}

	CRD bool wants_node() const { return bottom || ((cntA | cntB) == 0u && node != CRG_END); }
	CRD bool wants_instance() const { return !bottom && (cntA | cntB) != 0u; }

	/* one iteration of the flat loop; precondition: !done() */
	CRD void step(const DevScene &sc, TraceCounters *ctr) {
		if (bottom || (cntA | cntB) == 0u) node_step(sc, ctr);
		else instance_step(sc, ctr);
	}

	/* the tail of a bottom-level step: once the mesh BVH is exhausted, back to the top level (instance.c:175-184) */
	CRD void finish_bottom(const DevScene &sc) {
		if (node == CRG_END) {
			if (instHit) best.inst = curInst;
			bottom = false;
			o = wo; d = wd;
			rs = cr_ray_setup(o, d);
			base = sc.pairs + sc.top.pair_offset;
			node = topNext;
			spBase = 0;
		}
	}

	/* precondition: wants_node() */
	CRD void node_step(const DevScene &sc, TraceCounters *ctr) {
		{
			/* ---- one child-pair step (bvh.c:391-439) */
			const float4 *p4 = reinterpret_cast<const float4 *>(base + node);
			const float4 q0 = __ldg(p4 + 0), q1 = __ldg(p4 + 1), q2 = __ldg(p4 + 2);
			const uint4 q3 = __ldg(reinterpret_cast<const uint4 *>(p4 + 3));
			const float lb[6] = { q0.x, q0.y, q0.z, q0.w, q1.x, q1.y };
			const float rb[6] = { q1.z, q1.w, q2.x, q2.y, q2.z, q2.w };
			if (COUNT) ctr->pairs++;
			float tL, tR;
			const bool hitL = cr_node_test(lb, rs, o, best.t, tL);
			const bool hitR = cr_node_test(rb, rs, o, best.t, tR);
			const bool leafL = (q3.z & CRG_LEAF_BIT) != 0u, leafR = (q3.w & CRG_LEAF_BIT) != 0u;
			const bool goL = hitL && !leafL, goR = hitR && !leafR;
			uint32_t next;
			if (goL & goR) {
				const bool swap = tL > tR;                                         /* bvh.c:424-431 */
				next = swap ? q3.y : q3.x;
				stack[sp++] = swap ? q3.x : q3.y;
			} else if (goL ^ goR) {
				next = goL ? q3.x : q3.y;
			} else {
				next = (sp == spBase) ? CRG_END : stack[--sp];
			}
			if (bottom) {
				/* left leaf, then right leaf (bvh.c:402-418), as ONE loop so that lanes with a left leaf and lanes with a
				 * right leaf test their triangles together */
				const uint32_t nL = (hitL && leafL) ? (q3.z & ~CRG_LEAF_BIT) : 0u;
				const uint32_t nR = (hitR && leafR) ? (q3.w & ~CRG_LEAF_BIT) : 0u;
				node = next;
				if (nL + nR) instHit |= cr_leaf_tris2<COUNT>(tris, slotBase, q3.x, nL, q3.y, nR, o, d, best, ctr);
				finish_bottom(sc);
			} else {
				if (hitL && leafL) { pendA = q3.x; cntA = q3.z & ~CRG_LEAF_BIT; }
				if (hitR && leafR) { pendB = q3.y; cntB = q3.w & ~CRG_LEAF_BIT; }
				node = next;
			}
		}
	}

	/* precondition: wants_instance() */
	CRD void instance_step(const DevScene &sc, TraceCounters *ctr) {
		{
			/* ---- one instance of a pending top-level leaf (bvh.c:468-486) */
			uint32_t idx;
			if (cntA) { idx = pendA++; --cntA; } else { idx = pendB++; --cntB; }
			const int cur = __ldg(sc.top_prims + sc.top.slot_offset + idx);
			const DevInstance *inst = sc.instances + cur;
			const float4 *m4 = reinterpret_cast<const float4 *>(inst->Ainv);
			const float4 r0 = __ldg(m4 + 0), r1 = __ldg(m4 + 1), r2 = __ldg(m4 + 2);
			const float Ainv[12] = { r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w };
			const uint4 meta = __ldg(reinterpret_cast<const uint4 *>(&inst->kind));    /* kind, bvh, ray_offset, radius */
			v3 oo, od;
			cr_object_ray(Ainv, __uint_as_float(meta.z), wo, wd, oo, od);
			if (meta.x == CRS_INST_MESH) {                                         /* instance.c:169-175 */
				if (COUNT) ctr->insts++;
				const DevBvh *bvh = sc.bvhs + meta.y;
				const uint32_t nodeCount = __ldg(&bvh->node_count);
				const uint32_t slotOff = __ldg(&bvh->slot_offset);
				if (nodeCount < 1u) {
					best.inst = -1;                                                /* bvh.c:362-365 quirk */
				} else if (nodeCount == 1u) {                                      /* bvh.c:382-387 */
					const RaySetup ors = cr_ray_setup(oo, od);
					float rbnd[6], te;
					for (int k = 0; k < 6; ++k) rbnd[k] = __ldg(&bvh->root_bounds[k]);
					if (cr_node_test(rbnd, ors, oo, best.t, te))
						if (cr_leaf_tris<COUNT>(sc.tris + slotOff, slotOff, __ldg(&bvh->root_first), __ldg(&bvh->root_count), oo, od, best, ctr))
							best.inst = cur;
				} else {
					bottom = true;
					topNext = node;
					o = oo; d = od;
					rs = cr_ray_setup(o, d);
					base = sc.pairs + __ldg(&bvh->pair_offset);
					tris = sc.tris + slotOff;
					slotBase = slotOff;
					curInst = cur;
					instHit = false;
					spBase = sp;
					node = 0u;
				}
			} else {                                                               /* instance.c:45-51 */
				if (COUNT) ctr->spheres++;
				if (cr_sphere_test(oo, od, __uint_as_float(meta.w), best.t)) best.inst = cur;
			}
		}
	}
};

template <bool COUNT>
CRD Hit cr_closest_hit(const DevScene &sc, v3 wo, v3 wd, TraceCounters *ctr) {
	uint32_t stack[2 * CRG_MAX_STACK + 2];
	Traversal<COUNT> tr;
	tr.stack = stack;
	tr.begin(sc, wo, wd);
	while (!tr.done()) tr.step(sc, ctr);
	return tr.best;
}

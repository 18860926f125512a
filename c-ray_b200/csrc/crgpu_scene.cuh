/*
 * crgpu_scene.cuh — device-side scene layout (HBM) for the B200 hot path.
 *
 * Built once per scene by crgpu_scene_create() from the flat description (include/crscene.h).
 * The reference layout is pointer-linked AoS (struct bvhNode 32 B bvh.c:37-42, struct poly 40 B of
 * indices poly.h:11-18 into global vertex arrays, struct instance 160 B instance.h:23-28).  Here:
 *
 *   PairNode  64 B, 64-B aligned: BOTH children of one internal node (bounds + refs), because the
 *             traversal always fetches and tests the two children together (bvh.c:392-398).  One
 *             LDG.128 x4 per step instead of two dependent 32-B fetches; internal nodes are renumbered
 *             in BFS order, so the top of each tree is one contiguous range.
 *   PackedTri 48 B, 16-B aligned, in LEAF ORDER (indexed by primIndices slot, not by poly): v0, e1, e2
 *             and n = e1 x e2 precomputed with the reference's exact fp32 operations (poly.c:20-22), so
 *             a leaf's triangles are contiguous and the Möller–Trumbore test needs no index chasing.
 *   ShadePoly 80 B per poly: pre-gathered vertex normals / texcoords / material for the shade kernel.
 *   Instance  128 B: Ainv and A (3x4 rows each), kind, object parameters.
 */
#pragma once
/* limits of the device node interpreter (crgpu_shade.cuh), enforced at upload (crgpu_api.cu check_bsdf) */
#define CRG_NODE_DEPTH 3      /* color->value->color nesting of the hot interpreter (NodeEval: the node kinds JSON scenes contain) */
#define CRG_XNODE_DEPTH 8     /* edges below the first node of a kind only the complete interpreter knows (NodeX: SURVEY 8 f4) */
#define CRG_ADD_STACK 4       /* operand stack of nested ADD bsdfs */
#include <stdint.h>
#include "../../include/crscene.h"

#define CRG_LEAF_BIT 0x80000000u
#define CRG_MAX_STACK 64            /* MAX_BVH_DEPTH, bvh.c:32 */

struct __align__(64) PairNode {
	float lb[6];                    /* left child: minx,maxx,miny,maxy,minz,maxz */
	float rb[6];                    /* right child */
	uint32_t lref, rref;            /* internal child: its pair index; leaf child: first prim slot (local to the BVH) */
	uint32_t lmeta, rmeta;          /* CRG_LEAF_BIT | primCount for leaves, 0 for internal children */
};

struct __align__(16) PackedTri {
	float v0[3], e1[3], e2[3], n[3];
};

struct __align__(16) ShadePoly {
	float n0[3], n1[3], n2[3];      /* vertex normals (n0 = geometric normal when !has_normals) */
	float t0[2], t1[2], t2[2];      /* texture coordinates */
	uint32_t material;              /* global material index */
	uint32_t flags;                 /* bit0 has_normals, bit1 has_uv */
	uint32_t pad[3];
};

struct DevBvh {
	uint32_t pair_offset;           /* into pairs[] */
	uint32_t pair_end;              /* one past this BVH's last pair node */
	uint32_t node_count;            /* reference nodeCount (0, 1 or >1 select the code path, bvh.c:362-387) */
	uint32_t slot_offset;           /* into tris[] / slot_poly[] (mesh) or top_prims[] (top level) */
	uint32_t root_first, root_count;/* when node_count == 1: the root is a leaf */
	float    root_bounds[6];
	uint32_t pad;
};

struct __align__(16) DevInstance {
	float Ainv[12];
	float A[12];
	uint32_t kind;                  /* CRS_INST_SPHERE / CRS_INST_MESH */
	uint32_t bvh;                   /* mesh: index into bvhs[] */
	float    ray_offset;
	float    radius;                /* sphere */
	uint32_t material;              /* sphere: global material index */
	uint32_t pad[3];
};

struct DevMaterial {
	float emission[3];
	float IOR;
	int32_t bsdf;
	uint32_t flags;                 /* bit0: graph reads uv (image / checker nodes); bit1: emission != 0 */
	uint32_t pad[2];
};

struct DevTexture {
	uint32_t width, height, channels, is_float, has_alpha;
	uint32_t wmask, hmask;          /* width-1 / height-1 when that dimension is a power of two, else 0 (x % W == x & (W-1), also for the
	                                   2^64-wrapped negative coordinates of texture.c:34-35) */
	uint32_t pad;
	const uint8_t *data;
};

struct DevCamera {
	float sensor_x, sensor_y, aperture, focal_distance;
	float forward[3], right[3], up[3];
	int32_t width, height;
	float A[12];
};

struct DevScene {
	DevCamera cam;
	uint32_t image_width, image_height, sample_count, bounces;
	int32_t  background;
	uint32_t instance_count;
	DevBvh   top;
	const PairNode   *pairs;
	const PackedTri  *tris;
	const uint32_t   *slot_poly;    /* prim slot -> global poly index */
	const ShadePoly  *spolys;
	const int32_t    *top_prims;    /* top-level primIndices (instance indices) */
	const DevBvh     *bvhs;
	const DevInstance*instances;
	const DevMaterial*materials;
	const crs_node   *nodes;
	const DevTexture *textures;
	const float      *u8_to_unit;   /* [256]: (float)i / 255.0f, the byte→float division of texture.c:48-60 done once */
};

// Flattened, pointer-free scene layout shared by the host flattener and the CUDA kernels.
// See DESIGN.md "Data layout in HBM".
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#else
struct float4 { float x, y, z, w; };
struct float2 { float x, y; };
struct int4 { int x, y, z, w; };
struct uchar4 { unsigned char x, y, z, w; };
typedef unsigned long long cudaTextureObject_t;
#endif

namespace fw {

enum ShapeKind : int {
    SH_SPHERE = 0,    // objects/sphere.rs
    SH_RECT = 1,      // objects/rect.rs      (plane in i0 bits 0-1: 0 XY, 1 XZ, 2 YZ; flip_normal bit 2)
    SH_RECT3D = 2,    // objects/rect3d.rs    (i0 = first face ShapeRec, i1 = face count)
    SH_MESH = 3,      // objects/mesh.rs      (i0 = MeshRec index)
    SH_DISK = 4,      // objects/disk.rs
    SH_CYLINDER = 5,  // objects/cylinder.rs
    SH_CONE = 6,      // objects/cone.rs
    SH_MEDIUM = 7,    // objects/volume.rs    (i0 = inner ShapeRec, f[0] = density)
};
enum MatKind : int {  // material.rs; MAT_MISS is a queue id only
    MAT_LAMBERTIAN = 0, MAT_METAL = 1, MAT_DIELECTRIC = 2, MAT_EMISSIVE = 3, MAT_ISOTROPIC = 4, MAT_MISS = 5,
    MAT_NUM_QUEUES = 6
};
enum TexKind : int { TEX_CONSTANT = 0, TEX_CHECKER = 1, TEX_PERLIN = 2, TEX_TURBULENCE = 3, TEX_MARBLE = 4, TEX_IMAGE = 5 };
// Textures on the longest root-to-leaf path of one texture tree (CheckerTextures nest): texture_sample follows at most this many
// links, and the loader refuses deeper trees.
constexpr int FW_MAX_TEXTURE_DEPTH = 64;
enum EnvKind : int { ENV_COLOR = 0, ENV_SKY = 1, ENV_HDR = 2 };

// Linear-scan program (Renderer.use_bvh == false, scene.rs:137-149).  The scene's objects, in scene order, are
// compiled host-side into a short list of float4 words that travels in KERNEL PARAMETER space (constant bank):
// every lane of a warp is at the same item, so the words are fetched through the uniform datapath and the item
// switch is a uniform branch — no per-lane loads of object / shape records at all.  word0.y = type | plane << 8.
enum LinItem : int {   // one bit per type: the dispatch is a chain of bit tests, most frequent first
    LIN_END = 0,
    LIN_RECT = 1,      // 2 words: (k, type | plane << 8, obj, prim), (min1, min2, max1, max2)           (rect.rs:48-62)
    LIN_BOX6 = 2,      // 4 words: a Rect3d whose six faces are the canonical ones of Rect3d::new (rect3d.rs:18-80):
                       //          (lo.x, type, obj, lo.y), (lo.z, hi.x, hi.y, hi.z), padded box (lo.xyz, hi.x), (hi.y, hi.z, -, -)
    LIN_XFORM_T = 4,   // 1 word : (pos.x, type, pos.y, pos.z): current ray = (o - pos, d)              (scene.rs:250-252)
    LIN_XFORM_R = 8,   // 4 words: same, then 3 columns of inv_rotation_mat: both rotated                (scene.rs:246-249)
    LIN_SPHERE = 16,   // 1 word : (radius, type, obj, -)                                               (sphere.rs:32-50)
    LIN_GENERIC = 32,  // 1 word : (-, type, obj, -): any other object, through object_test on the world ray
};
constexpr int LIN_SPACE_HAS_RECTS = 0x100;  // on XFORM items: rectangle items follow in this space (set up the shared division)
constexpr int FW_LIN_MAX_WORDS = 160;   // 2.5 KiB of the 4 KiB kernel-parameter space
struct LinProgram {
    float4 w[FW_LIN_MAX_WORDS];
};

constexpr int OBJ_KIND_MASK = 0xff;
constexpr int OBJ_ROTATED = 1 << 8;   // cos_trace < 0.999 (scene.rs:242-246): ray is rotated into object space
constexpr int OBJ_FLIP = 1 << 9;      // RenderObject.flip_normals (scene.rs:259-261)
constexpr int OBJ_MESH_ORD_SHIFT = 16; // bits 16..20: ordinal of a top-level TriangleMesh object among the scene's meshes (0..7; walk kernels)
constexpr int FW_MAX_WALK_MESHES = 8;  // top-level meshes a scene may have for the mesh-entry path (else: lock-step pass 2)

struct ShapeRec {  // 48 B
    int kind, material, i0, i1;
    float f[8];
};
struct MeshRec {  // 64 B
    int root_code;   // wide node index (>= 0) or leaf code (< 0) of this mesh's BVH root
    int tri_first;   // first triangle slot (triangles are stored in BVH leaf order)
    int tri_count;
    int flags;       // bit0 has_normals, bit1 has_uvs
    int material;
    int pad[3];
    float lo[4], hi[4];  // the root's box (bvh.rs:117 tests it first)
};
struct MatRec {  // 32 B
    int kind, tex;
    float param;
    int needs_uv;   // 1 if the material's texture tree contains an ImageTexture (the only uv consumer)
    float albedo[3], pad1;
};
struct TexRec {  // 32 B
    int kind, a, b, depth;   // checker: a = odd, b = even; image: a = image index
    float scale;
    float color[3];
};
struct ImageRec {  // 16 B
    cudaTextureObject_t tex;  // uchar4 point-sampled, unnormalised coordinates
    uint32_t w, h;
};
struct EnvRec {
    int kind;
    uint32_t w, h;
    int pad;
    float a[4];               // ColorEnv colour | SkyEnv zenith
    float b[4];               // SkyEnv horizon
    cudaTextureObject_t tex;  // HdrEnvironment: float4 point-sampled
};

// BVH: the LEAVES are those of the reference's binary median-split tree (bvh.rs:21-71: same items, same boxes, same
// DFS order); the hierarchy above them is rebuilt with a surface-area heuristic and collapsed into 4-wide nodes
// (scene_host.cpp build_bvh explains why that cannot change which items a ray tests).
// Wide node = 8 x float4 (128 B, one cache line, 128-byte aligned):
//   [0..2] child min x / y / z (one lane per child)   [3..5] child max x / y / z
//   [6]    child codes (int bits):  >= 0 wide node index;  < 0 leaf: p = ~code, items [p >> 1, (p >> 1) + (p & 1) + 1)
//          of the tree's item list (1 or 2 items: bvh.rs Leaf / DoubleLeaf); empty slots carry an inverted box
//   [7]    host-side bookkeeping only (which children hold a Disk); the kernels do not read it
struct DeviceScene {
    const float4* nodes;       // wide nodes of all trees (top-level tree first)
    float4 top_lo, top_hi;     // the top-level root's box; top_lo.w = asfloat(root code)
    const float4* top_leaves;  // 2 per top-level leaf, DFS order: (box min, asfloat(first rank)), (box max, asfloat(item count))
    int n_top_leaves;
    const int* top_items;      // object ids in top-level DFS leaf order (rank = tie-break key, bvh.rs:128,141)
    const float4* leaf_posr;   // obj_posr reordered by top-level DFS leaf rank (no indirection in the leaf loop)
    const int4* leaf_meta;     // obj_meta reordered by rank; .w = object id
    const float4* obj_posr;    // per object: (position.xyz, sphere radius or 0)
    const int4* obj_meta;      // per object: (kind | flags, material, shape index, 0)
    const float4* obj_rot;     // per object: 3 x float4 = columns of rotation_mat
    const float4* obj_irot;    // per object: 3 x float4 = columns of inv_rotation_mat
    const ShapeRec* shapes;
    const MeshRec* meshes;
    const float4* tri_verts;   // per triangle slot: 3 x float4 (p0, p1, p2; p0.w = asfloat(original index))
    const float4* tri_perm;    // 3 copies of tri_verts, copy kz holds every vertex as (v[kx], v[ky], v[kz]) for the dominant
                               // axis kz of mesh.rs:146-153 (kx = kz+1, ky = kx+1 mod 3): [(kz * n_tris + slot) * 3 + vertex]
    const float4* tri_normals; // per triangle slot: 3 x float4 (only for meshes with normals; else unused)
    const float2* tri_uvs;     // per triangle slot: 3 x float2 (default (0,0),(1,0),(0,1) if the mesh has none)
    const MatRec* mats;
    const TexRec* texs;
    const ImageRec* images;
    EnvRec env;
    int n_objects;
    int n_nodes;
    int n_tris;                // triangle slots of all meshes (stride of tri_perm's copies)
    int top_root_is_valid;     // 0 if the top-level BVH was not built (linear scenes may still build it)
    int has_medium;
    int has_unbounded;         // some top-level item's box does not bound its geometry (Disk): node flags matter
    // Closest-hit answer for a ray whose direction is NaN in all three components (see nan_direction_winner):
    // object id (-1 = miss) and primitive (mesh: last triangle slot, Rect3d: last face), for BVH and linear roots.
    int nan_bvh_obj, nan_bvh_prim, nan_lin_obj, nan_lin_prim;
    int mesh_rank[FW_MAX_WALK_MESHES];   // top-level DFS rank of the mesh object with ordinal k (scenes with <= 8 top-level meshes)
    int mesh_root[FW_MAX_WALK_MESHES];   // ... the root (wide node) of its triangle tree
    int mesh_tri0[FW_MAX_WALK_MESHES];   // ... its first triangle slot
};

struct CameraRec {  // camera.rs:7-16
    float position[3], horizontal[3], vertical[3], lower_left[3], u[3], v[3], w[3];
    float lens_radius;
};

}  // namespace fw

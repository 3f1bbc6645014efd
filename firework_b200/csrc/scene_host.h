// Host side of the drop-in boundary: firework serde-YAML scene document -> neutral description ->
// BVHs built with the reference's split rule -> pointer-free flattened arrays (fw_types.h).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "fw_types.h"

namespace fw {

struct V3 {
    float x, y, z;
};
struct Box {
    V3 mn, mx;
};

struct AssetDesc {
    std::string path;
    int kind = 0;  // 0 = RGBA8 image (ImageTexture), 1 = fp32 RGB equirect map (HdrEnvironment)
    uint32_t w = 0, h = 0;
    std::vector<uint8_t> rgba;  // kind 0
    std::vector<float> rgb;     // kind 1
    bool provided = false;
};

struct MeshDesc {  // objects/mesh.rs:12-19
    std::vector<uint32_t> indicies;
    std::vector<V3> verts;
    bool has_normals = false, has_uvs = false;
    std::vector<V3> normals;
    std::vector<float> uvs;  // 2 per vertex
    int material = 0;
};

struct ObjectDesc {  // scene.rs:268-277
    int shape = 0;
    V3 position{0, 0, 0};
    float rotor[4] = {1, 0, 0, 0};  // s, xy, xz, yz
    bool flip_normals = false;
};

struct SceneDesc {
    std::vector<TexRec> texs;
    std::vector<MatRec> mats;
    std::vector<ShapeRec> shapes;
    std::vector<MeshDesc> meshes;
    std::vector<ObjectDesc> objects;
    std::vector<AssetDesc> assets;
    int env_kind = ENV_COLOR;
    float env_a[3] = {0, 0, 0}, env_b[3] = {0, 0, 0};
    int env_asset = -1;
};

// Parses a firework scene document (the output of serde_yaml::to_string(&Scene)). Unknown tags are errors.
bool load_scene_yaml(const char* text, size_t len, SceneDesc& out, std::string& err);

// One BVH in flattened form (see fw_types.h for the node encoding).
struct FlatBVH {
    std::vector<float4> nodes;   // 8 float4 per WIDE node (fw_types.h), child links local to this tree
    std::vector<int> items;      // item ids in DFS leaf order
    Box root_box{};              // the binary root's box (bvh.rs:117 tests it before anything else)
    int root_code = 0;           // wide node index (>= 0) or leaf code (< 0) of the root
    int max_depth = 0;           // depth of the reference's binary tree
    int wide_depth = 0;          // depth of the collapsed 4-wide tree
};
// The reference's median split (bvh.rs:21-71): stable sort on centroid[depth % 3], leaves of 1 or 2.
// `item_unbounded` (optional, same length as item_boxes) marks items whose box does NOT bound their geometry
// (Disk: disk.rs:85-90); every node above such an item is flagged so the traversal never distance-culls it.
// device < 0 builds on the host; otherwise the sorts and the SAH splits run on that CUDA device (kernels_build.cu) and
// the result is the host's, byte for byte.  Returns FW_OK or the FW_ERR_* code of `err`.
int build_bvh_on(int device, const std::vector<Box>& item_boxes, FlatBVH& out, std::string& err,
                 const std::vector<uint8_t>* item_unbounded = nullptr);
// The tree flatten_scene builds: on the device of the calling thread's innermost BvhDeviceScope when it has at least
// kDeviceBvhMinItems items, else on the host.
bool build_bvh(const std::vector<Box>& item_boxes, FlatBVH& out, std::string& err,
               const std::vector<uint8_t>* item_unbounded = nullptr);
// While alive, lets the calling thread's build_bvh calls build large trees on `device` (< 0: host), and records the
// FW_ERR_* code of a failed build (FW_ERR_CUDA for a device failure) in `code`.  fw_scene_commit sets one around
// flatten_scene, which therefore does not know where its trees are built.
struct BvhDeviceScope {
    explicit BvhDeviceScope(int device);
    ~BvhDeviceScope();
    BvhDeviceScope(const BvhDeviceScope&) = delete;
    BvhDeviceScope& operator=(const BvhDeviceScope&) = delete;
    int device;
    int code = -2;   // FW_ERR_SCENE
    BvhDeviceScope* prev;
};

// fw_scene_commit builds a tree of at least this many items on its device (DESIGN.md §8: measured crossover).
constexpr size_t kDeviceBvhMinItems = 8192;

// Device stages of build_bvh (kernels_build.cu).  bvh_leaf_order_device: the item order of the median-split tree, and
// whether some node met a NaN centroid on its axis.  bvh_sah_device: the SAH interior over leaves with the given boxes
// and item counts (DFS order); records in level order, parents before children, record 0 the root (no records when
// there is one leaf); leaf_order is the final leaf permutation.
struct SahRec {
    int depth;
    int left, right;   // record index (>= 0), or ~position of a single leaf in leaf_order
    int k;             // leaves on the left
};
bool bvh_leaf_order_device(int device, const std::vector<Box>& boxes, std::vector<int>& order, bool& nan, std::string& err);
bool bvh_sah_device(int device, const std::vector<Box>& leaf_boxes, const std::vector<int>& leaf_counts, int max_depth,
                    std::vector<SahRec>& recs, std::vector<int>& leaf_order, std::string& err);

struct HostFlat {
    std::vector<float4> nodes;
    std::vector<int> top_items;
    std::vector<float4> top_leaves;   // 2 per top-level leaf in DFS order: (box min, asfloat(first rank)), (box max, asfloat(items))
    std::vector<float4> lin_words;  // linear-scan program (fw_types.h LinItem), END-terminated
    bool lin_generic = false;       // the program contains LIN_GENERIC items
    int lin_rect_tests = 0;         // AARect::hit calls per ray in the program (RECT items + 6 per BOX6)
    std::vector<float4> obj_posr, leaf_posr;
    std::vector<int4> obj_meta, leaf_meta;
    std::vector<float4> obj_rot, obj_irot;
    std::vector<Box> obj_aabb;  // world boxes (scene.rs:167-212), kept for tests / stats
    std::vector<ShapeRec> shapes;
    std::vector<MeshRec> meshes;
    std::vector<float4> tri_verts, tri_normals, tri_perm;
    std::vector<float2> tri_uvs;
    std::vector<MatRec> mats;
    std::vector<TexRec> texs;
    int top_depth = 0;
    int top_nodes = 0;
    Box top_root_box{};
    int top_root_code = 0;
    bool has_medium = false;
    bool has_unbounded = false;
    int nan_bvh_obj = -1, nan_bvh_prim = 0, nan_lin_obj = -1, nan_lin_prim = 0;
    bool has_mesh = false;          // some object is (or wraps) a TriangleMesh
    bool has_top_mesh = false;      // some render object IS a TriangleMesh
    bool has_medium_mesh = false;   // some ConstantMedium wraps a TriangleMesh
    // Collect / test walk kernels (walk.cuh): usable when both roots are wide nodes, the per-lane stack bounds hold, the
    // scene has few enough top-level meshes for the entry queue, and (t, rank, primitive) packs into one 64-bit key.
    int top_wide_depth = 0, mesh_wide_depth = 0;
    int n_top_meshes = 0;           // render objects that ARE a TriangleMesh
    int mesh_rank[FW_MAX_WALK_MESHES] = {0, 0, 0, 0, 0, 0, 0, 0};   // DFS rank of the mesh object with ordinal k
    int walk_prim_bits = 0;         // key = t bits << 32 | ~rank << prim_bits | ~prim
    bool walk_ok = false;
};
bool flatten_scene(const SceneDesc& desc, HostFlat& out, std::string& err);

struct RenderParamsHost {
    uint32_t width, height, samples, sample_begin, sample_count, use_bvh;
    float gamma;
    float cam_pos[3], look_at[3];
    float vfov, aperture, focus_dist;
    uint64_t seed;
};
CameraRec make_camera(const RenderParamsHost& p);

// Records the message fw_last_error() returns on this thread and passes `code` through (api.cu).
int set_last_error(int code, const std::string& msg);

}  // namespace fw

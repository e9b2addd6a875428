// rtp_internal.h — structures shared by the host layer (rtp_host.cpp) and the device layer
// (rtp_device.cu). Not part of the ABI.
#pragma once

#include <cstddef>
#include <cstdint>
#include <limits>
#include <string>
#include <vector>

#include "../../include/rtp.h"

namespace rtp {

// ---------------------------------------------------------------------------------------------
// Device layout (HBM). All records are 16-byte aligned so they load as 128-bit vectors.
//
// Nodes are stored in the reference's depth-first, left-before-right order (pre-order), so the
// reference traversal bvh.rs:93-119 becomes a stack-free walk: a node that passes its slab test
// is followed by node+1 (its left child, or for a leaf simply the next subtree), a node that
// fails jumps to `skip`, the first pre-order index after its subtree.
// ---------------------------------------------------------------------------------------------

constexpr uint32_t kNoPrim = 0xFFFFFFFFu;

struct alignas(64) DNode {  // 64 B
    double bmin[3];
    double bmax[3];
    uint32_t skip;  // pre-order index of the next node once this subtree is done
    uint32_t prim;  // leaf: primitive slot (= DFS rank of the leaf); branch: kNoPrim
    uint32_t kind;  // leaf: rtp_hittable_kind
    uint32_t _pad;  // List roots: 1 = test the box in DPrim first (a leaf of a nested Bvh), 0 = no gate (hittable.rs:110-120)
};
static_assert(sizeof(DNode) == 64, "DNode must be 64 bytes");

// One primitive per leaf (bvh.rs:43-47), stored in DFS-rank order so a traversal touches them
// in increasing address order. Triangle: a, ba = a-b, ca = a-c precomputed on the host with the
// same IEEE subtraction the reference performs per test (hittable.rs:71-72) — bit-identical.
// Sphere: center in a[], radius in ba[0]. The leaf's own exact f64 box (the reference's per-leaf
// slab gate, bvh.rs:96) travels with the primitive so gate + test need one 128-byte record.
struct alignas(16) DPrim {  // 128 B
    double a[3];
    double ba[3];
    double ca[3];
    uint32_t leaf;      // LeafId handed back to the caller
    uint32_t material;  // MaterialId
    double bmin[3];
    double bmax[3];
};
static_assert(sizeof(DPrim) == 128, "DPrim must be 128 bytes");

// Culling tree in f32: a 4-wide tree over the rank-ordered leaf sequence. A node holds the boxes of its (up to) four
// children, in rank order, as six 4-lane planes (structure of arrays), so one 128-byte line answers four slab tests and a
// ray picks its near / far planes by ADDRESS (offset 0 or 16 inside each axis block) instead of by select. Every child box is
// the child's exact f64 box rounded OUTWARD and inflated by 2^-21 * max(|min|,|max|) per axis, so that an f32 slab
// evaluation with the matching ray-side slack is a rigorous lower / upper bound of the reference's f64 evaluation
// (rtp_device.cu collide32; DESIGN.md §4). child[k]: internal = index of the child node; leaf = kWideLeaf | kind << 30 |
// kWideBig if big | primitive slot; unused = kWideEmpty with an inverted (+inf, -inf) box that no ray can enter.
constexpr uint32_t kWideLeaf = 0x80000000u;
constexpr uint32_t kWideBig = 0x20000000u;       // leaf child word: the primitive is one of the scene's big primitives (trace_any_kernel tests those up front)
constexpr uint32_t kWideSlotMask = 0x1FFFFFFFu;  // leaf child word: primitive slot
constexpr uint32_t kWideEmpty = 0xFFFFFFFFu;
struct alignas(128) DWide {  // 128 B = one L1/L2 line
    float plane[3][2][4];    // [axis][0 = min, 1 = max][child]
    uint32_t child[4];
    uint32_t _pad[4];
};
static_assert(sizeof(DWide) == 128, "DWide must be 128 bytes");

// Shading attributes of a triangle (mesh.rs:7-11 normals/uvs of its three vertices), read once
// per accepted path vertex, never during traversal.
struct alignas(16) DAttr {  // 128 B; uv first so that both arrays start 16-byte aligned
    double uv[3][2];
    double n[3][3];
    double _pad;
};
static_assert(sizeof(DAttr) == 128, "DAttr must be 128 bytes");

struct DTexture {
    uint32_t kind;
    uint32_t width, height;
    uint32_t odd, even;
    uint32_t _pad;
    int64_t seed;
    double rgb[3];
    const uint8_t* rgba;  // device pointer
};

struct DMaterial {
    uint32_t scatter, absorb, absorb_texture, emit_kind;
    uint32_t emit_texture, _pad[3];
    double scatter_param;
    double absorb_rgb[3];
    double emit_rgb[3];
};

struct DSceneView {  // passed by value to kernels
    const DNode* nodes;
    const DWide* wide;
    const double* wide_boxes;  // [node][child][min xyz, max xyz] exact f64 child boxes (counting kernels: violation check)
    const DWide* any_wide;     // the tree the any-order lanes walk: `wide`, or the order-free tree of a big scene
    const double* any_boxes;
    const DPrim* prims;
    const DAttr* attrs;
    const DMaterial* materials;
    const DTexture* textures;
    uint32_t n_nodes;
    uint32_t n_prims;
    uint32_t root_kind;
    uint32_t bg_kind;
    uint32_t bg_texture;
    uint32_t f32_culling;  // 1: scene magnitudes allow the f32 conservative slab test
    double bg_rgb[3];
    // any-order walk (DESIGN.md §4b): front-to-back traversal with distance culling, exact because every leaf that can matter is
    // still tested and the rare ray whose answer could depend on the reference's visiting order is re-walked in order
    uint32_t any_order;    // 1: eligible rays of this scene use it
    uint32_t any_cap;      // entries of the per-lane any-order stack
    uint32_t n_big;        // primitives exempt from distance culling (the outsized ones: extent above 16x the median), at most kMaxBig
    uint32_t fast_slab;    // 1: every box is finite and ordered, so eligible rays may use the sign-selected slab test (collide_fast)
    uint32_t big[8];       // their slots | kind << 31
    double any_E;          // largest box extent of a triangle that is not big
    double any_A;          // largest |coordinate| of such a triangle
    float any_Ef, any_Af;  // the same, rounded up to f32
    float any_Cf, any_Rf;  // spheres that are not big: largest |centre coordinate| and radius, rounded up; any_Rf < 0: there are none
    float cull[6];         // culled-set box: the union of the leaf boxes that are not big, rounded out like a DWide child box (min xyz,
                           // max xyz); a ray whose window closes before it is done after its big-primitive tests. Empty: (+inf, -inf)
};
constexpr uint32_t kMaxBig = 8;

// ---------------------------------------------------------------------------------------------
// Host-side flattened scene produced by rtp_host.cpp and uploaded by rtp_device.cu
// ---------------------------------------------------------------------------------------------
// Big arrays that were BUILT on a device (rtp_build.cu device_build_scene) and never existed on the host: device_scene_upload
// adopts them on that device and copies them peer to peer to the other devices of a multi-device scene.
struct DevArrays {
    bool valid = false;
    mutable bool adopted = false;  // the replica on `device` owns the arrays now (device_scene_upload); the others copied from them
    int device = -1;
    DNode* nodes = nullptr; size_t n_nodes = 0;
    DWide* wide = nullptr; double* wide_boxes = nullptr; size_t n_wide = 0;
    DPrim* prims = nullptr; DAttr* attrs = nullptr; size_t n_prims = 0;
};

struct FlatScene {
    DevArrays dev;
    size_t prim_count() const { return dev.valid ? dev.n_prims : prims.size(); }
    size_t node_count() const { return dev.valid ? dev.n_nodes : nodes.size(); }
    size_t wide_count() const { return dev.valid ? dev.n_wide : wide.size(); }
    std::vector<DNode> nodes;
    std::vector<DWide> wide;
    std::vector<double> wide_boxes;
    uint32_t wide_depth = 0;         // nodes on the longest root-to-leaf path of the 4-wide tree
    std::vector<DPrim> prims;
    std::vector<DAttr> attrs;
    std::vector<DMaterial> materials;
    std::vector<DTexture> textures;            // rgba = nullptr here; filled at upload
    std::vector<std::vector<uint8_t>> images;  // per texture (empty unless Image)
    std::vector<uint32_t> leaf_order;          // LeafId by DFS rank
    uint32_t root_kind = 0;
    uint32_t depth = 0;              // of the reference tree (bvh.rs), what rtp_scene_info reports
    uint32_t n_reference_nodes = 0;  // 2n-1
    uint32_t device_depth = 0;       // of the culling tree the kernels walk
    bool list_gates = false;         // List root with nested Bvh items: some primitives are gated by a box (DNode::_pad)
    bool any_ok = false;             // the any-order walk may be used on this scene (prepare_any_order, rtp_host.cpp)
    std::vector<DWide> free_wide;    // second culling tree over the Morton order of the leaves (any-order walk of big scenes); may be empty
    std::vector<double> free_boxes;
    uint32_t free_depth = 0;
    uint32_t n_big = 0;
    uint32_t big[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    double any_E = 0.0, any_A = 0.0, any_C = 0.0, any_R = 0.0;
    bool any_spheres = false;        // some sphere is not big: the slack bound needs the sphere term
    float cull[6] = {std::numeric_limits<float>::infinity(), std::numeric_limits<float>::infinity(), std::numeric_limits<float>::infinity(),
                     -std::numeric_limits<float>::infinity(), -std::numeric_limits<float>::infinity(), -std::numeric_limits<float>::infinity()};  // DSceneView::cull
    double scene_mag = 0.0;    // largest |coordinate| of any node box
    bool boxes_finite = true;  // every box is finite and ordered (min <= max): precondition of the sign-selected slab test, of the
                               // f32 culling walk and of re-shaping the tree; otherwise the reference topology and the literal test are used
    rtp_emit background{};
};

// error plumbing (rtp_host.cpp)
int set_error(int code, const std::string& msg);

// The library's RTP_* environment switches (INTEGRATION.md), all read by read_switches (rtp_host.cpp) and parsed one way: a 0/1
// switch is on when it is set and atoi of its value is not 0, a number is clamped to its range, a word is compared exactly. A
// scene reads them once when it is created and keeps them; rtp_bvh_build_order and rtp_bvh_culled_set read them when called.
// RTP_PATH_BUDGET is the one switch read per render call (read_path_budget), so that a scene's frames may be split differently.
struct Switches {
    bool any_order = true;          // RTP_TRAVERSAL: "inorder" keeps every ray in the reference's visiting order
    bool f32_culling = true;        // RTP_F32_CULLING=0: exact f64 slab tests at every node, and no any-order walk
    bool simple_trace = false;      // RTP_TRACE_KERNEL=simple: one thread per ray
    bool simple_render = false;     // RTP_RENDER_KERNEL=simple: one thread per path
    bool reference_tree = false;    // RTP_TREE=reference: keep the median-split topology on the device
    int free_tree = -1;             // RTP_FREE_TREE 0 / 1; -1 (unset): scenes below 262,144 leaves get the order-free tree
    int device_build = -1;          // RTP_DEVICE_BUILD 0 / 1; -1 (unset): scenes of at least 65,536 leaves are built on the device
    uint32_t any_cap = 0;           // RTP_ANY_CAP, 4..48 entries of the any-order stack; 0 (unset): from the tree's depth
    bool any_setup_cull = true;     // RTP_ANY_SETUP_CULL=0: every any-order ray walks
    uint32_t tail_threshold = 65536;  // RTP_TAIL_THRESHOLD: a launch of at most this many paths runs in tail mode (0 = never)
    uint32_t chunk_log2 = 18;       // RTP_CHUNK_LOG2, 10..24: a host-buffer batch goes to the device in chunks of 2^this rays
    bool build_timing = false;      // RTP_BUILD_TIMING: phase times of the scene build on stderr
    bool debug_sync = false;        // RTP_DEBUG_SYNC: synchronise after every integrator launch
    bool lane_stats = false;        // RTP_LANE_STATS: lane occupancy of counted calls on stderr
};
Switches read_switches();
size_t read_path_budget();  // RTP_PATH_BUDGET, 1..2^31 paths per integrator launch; 0: unset

// An exact f64 box as the f32 culling box of a DWide child: rounded outward and inflated by 2^-21 * max(|min|, |max|) per axis
// (DESIGN.md §4; rtp_host.cpp)
void round_out(const double* bmin, const double* bmax, float* lo, float* hi);
// DSceneView::cull of the union [lo, hi] of the leaf boxes that are not big; lo > hi: there are none
void culled_set_box(const double* lo, const double* hi, float* cull);

// The any-order walk's second, order-free culling tree (prepare_any_order, rtp_host.cpp): RTP_FREE_TREE, or by default every scene
// below kFreeTreeLeaves leaves, gets one
constexpr size_t kFreeTreeLeaves = 262144;
inline bool want_free_tree(const Switches& sw, size_t n_leaves) { return sw.free_tree >= 0 ? sw.free_tree != 0 : n_leaves < kFreeTreeLeaves; }
// Builds that tree over the primitives that are not big into out->free_wide / free_boxes / free_depth; out->n_big is set. Slot s has
// the leaf box bmin[s * stride + k], bmax[s * stride + k] (k = 0..2), kind[s] and is_big[s]. Both scene builds call it.
void build_free_tree(const double* bmin, const double* bmax, size_t stride, const std::vector<uint8_t>& kind, const std::vector<uint8_t>& is_big,
                     FlatScene* out);

// host layer
// device_build: build a large flat Bvh scene on the GPU (rtp_build.cu device_build_scene); host-only callers pass false
int flatten_scene(const rtp_scene_desc* desc, const Switches& sw, FlatScene* out, bool device_build = false);

// device layer (rtp_device.cu, rtp_build.cu)
struct DeviceScene;
int ensure_device();  // binds device 0 if rtp_init has not been called; RTP_ERR_CUDA without a usable sm_100 GPU
// the reference's leaf order on the device: d_boxes n x {min xyz, max xyz}, d_order_out item index by DFS rank (device pointers)
int device_reference_order_dev(const double* d_boxes, uint32_t n, uint32_t* d_order_out);
// The whole of flatten_scene's geometry part on the current device for a flat (un-nested) Bvh scene: leaf boxes, the reference's
// depth-first order, the SAH culling tree over that order, primitive / attribute records, the 4-wide collapse and the any-order
// tables; then the host's order-free tree when want_free_tree asks for it. Fills out->dev and the host-side metadata. Returns RTP_OK, a negative status, or 1 = "not applicable, use the host
// path" (irregular boxes). sw.build_timing: phase times on stderr.
int device_build_scene(const rtp_scene_desc* d, const Switches& sw, FlatScene* out);
void device_free_arrays(DevArrays* a);
int device_scene_upload(const FlatScene& flat, const Switches& sw, int device /* < 0: the bound device */, DeviceScene** out);
void device_scene_free(DeviceScene* ds);
uint64_t device_scene_bytes(const DeviceScene* ds);

}  // namespace rtp

struct rtp_scene {
    rtp::FlatScene flat;  // nodes/prims/attrs are released after upload; leaf_order is kept
    rtp::DeviceScene* dev = nullptr;          // devs[0]: the device the *_device entry points use
    std::vector<rtp::DeviceScene*> devs;      // one replica per device of rtp_scene_create_multi's mask
    uint32_t n_leaves = 0, n_nodes = 0;
};

// rtp_build.cu — device side of `Bvh::new` (bvh.rs:36-91): the reference's depth-first leaf order computed on the GPU.
//
// make_bvh (bvh.rs:36-56) sorts a range by the AABB-centroid key of one axis (bvh.rs:58-67), cuts it at len/2 and recurses
// with the next axis; the axis depends only on the depth. All ranges of one depth are therefore sorted by the same axis,
// and the whole recursion is a loop over depths, each depth one segmented sort of ALL leaves by (range, key, LeafId)
// (ties by LeafId: the deterministic order shared with the host build and the oracle, DESIGN.md §2). The segmented sort is
// three stable LSD passes — LeafId, then the 64-bit order-preserving image of the f64 key, then the range's start position —
// done with cub::DeviceRadixSort (CUDA toolkit; library code, used for this once-per-scene stage only). The kernels here
// compute keys and split the ranges. Output: item index by rank, bit-identical to the host Builder (tests/test_gpu_parity.py).
#include <cuda_runtime.h>

#include <cub/device/device_radix_sort.cuh>

#include <cstdint>
#include <string>

#include "rtp_internal.h"

namespace rtp {

#define RTP_CUDA_B(expr)                                                                             \
    do {                                                                                             \
        cudaError_t _e = (expr);                                                                     \
        if (_e != cudaSuccess) { cudaGetLastError(); cleanup(); return set_error(RTP_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); } \
    } while (0)

// keys of one depth: the item's LeafId (== its index: items arrive in LeafId order) and the sortable image of its centroid key
__global__ void __launch_bounds__(256) build_keys_kernel(const double* __restrict__ boxes, const uint32_t* __restrict__ perm, uint32_t n, int axis,
                                                          unsigned long long* __restrict__ key64) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* b = boxes + static_cast<size_t>(perm[i]) * 6;
    double key = 0.5 * (b[axis] + b[3 + axis]);  // bvh.rs:61-62
    key = key + 0.0;                             // -0.0 and +0.0 compare equal in partial_cmp: one image for both
    unsigned long long u = static_cast<unsigned long long>(__double_as_longlong(key));
    u = (u >> 63) ? ~u : (u | 0x8000000000000000ull);  // monotone map f64 -> u64 (no NaN: rejected by the host validation)
    key64[i] = u;
}

__global__ void __launch_bounds__(256) build_segkeys_kernel(const uint32_t* __restrict__ perm, const uint32_t* __restrict__ start_of_item, uint32_t n,
                                                             uint32_t* __restrict__ segkey) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) segkey[i] = start_of_item[perm[i]];
}

// bvh.rs:64: the left half gets len/2 items. Position i holds item perm[i] of the range [start, start+len).
__global__ void __launch_bounds__(256) build_split_kernel(const uint32_t* __restrict__ perm, uint32_t n, uint32_t* __restrict__ start_of_item,
                                                           uint32_t* __restrict__ len_of_item) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t item = perm[i];
    const uint32_t s = start_of_item[item], l = len_of_item[item];
    if (l <= 1) return;
    const uint32_t half = l / 2;
    if (i - s < half) {
        len_of_item[item] = half;
    } else {
        start_of_item[item] = s + half;
        len_of_item[item] = l - half;
    }
}

__global__ void __launch_bounds__(256) build_init_kernel(uint32_t n, uint32_t* __restrict__ perm, uint32_t* __restrict__ start_of_item,
                                                          uint32_t* __restrict__ len_of_item) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    perm[i] = i; start_of_item[i] = 0; len_of_item[i] = n;
}

// boxes and the resulting order (item index by DFS rank) both live on the device
int device_reference_order_dev(const double* d_boxes, uint32_t n, uint32_t* d_order_out) {
    uint32_t *d_perm[2] = {nullptr, nullptr}, *d_k32[2] = {nullptr, nullptr}, *d_start = nullptr, *d_len = nullptr;
    unsigned long long* d_k64[2] = {nullptr, nullptr};
    void* d_temp = nullptr;
    auto cleanup = [&]() {
        cudaFree(d_perm[0]); cudaFree(d_perm[1]); cudaFree(d_k32[0]); cudaFree(d_k32[1]); cudaFree(d_start); cudaFree(d_len);
        cudaFree(d_k64[0]); cudaFree(d_k64[1]); cudaFree(d_temp);
    };
    if (n == 0) return RTP_OK;
    for (int k = 0; k < 2; ++k) {
        RTP_CUDA_B(cudaMalloc(reinterpret_cast<void**>(&d_perm[k]), static_cast<size_t>(n) * 4));
        RTP_CUDA_B(cudaMalloc(reinterpret_cast<void**>(&d_k32[k]), static_cast<size_t>(n) * 4));
        RTP_CUDA_B(cudaMalloc(reinterpret_cast<void**>(&d_k64[k]), static_cast<size_t>(n) * 8));
    }
    RTP_CUDA_B(cudaMalloc(reinterpret_cast<void**>(&d_start), static_cast<size_t>(n) * 4));
    RTP_CUDA_B(cudaMalloc(reinterpret_cast<void**>(&d_len), static_cast<size_t>(n) * 4));
    size_t temp_bytes = 0, need = 0;
    cub::DoubleBuffer<uint32_t> kb32(d_k32[0], d_k32[1]), vb(d_perm[0], d_perm[1]);
    cub::DoubleBuffer<unsigned long long> kb64(d_k64[0], d_k64[1]);
    RTP_CUDA_B(cub::DeviceRadixSort::SortPairs(nullptr, need, kb64, vb, static_cast<int>(n), 0, 64));
    temp_bytes = need;
    RTP_CUDA_B(cub::DeviceRadixSort::SortPairs(nullptr, need, kb32, vb, static_cast<int>(n), 0, 32));
    temp_bytes = need > temp_bytes ? need : temp_bytes;
    RTP_CUDA_B(cudaMalloc(&d_temp, temp_bytes));

    const unsigned grid = (n + 255) / 256;
    build_init_kernel<<<grid, 256>>>(n, vb.Current(), d_start, d_len);
    RTP_CUDA_B(cudaGetLastError());
    int seg_bits = 1;
    while ((1ull << seg_bits) < n) ++seg_bits;  // range start positions are < n
    int axis = 0;
    for (uint64_t longest = n; longest > 1; longest = (longest + 1) / 2, axis = (axis + 1) % 3) {
        // pass 1 (least significant): LeafId. The value array IS the id, so sort it as keys carrying itself.
        RTP_CUDA_B(cudaMemcpyAsync(kb32.Current(), vb.Current(), static_cast<size_t>(n) * 4, cudaMemcpyDeviceToDevice));
        RTP_CUDA_B(cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, kb32, vb, static_cast<int>(n), 0, seg_bits));
        // pass 2: centroid key of this depth's axis
        build_keys_kernel<<<grid, 256>>>(d_boxes, vb.Current(), n, axis, kb64.Current());
        RTP_CUDA_B(cudaGetLastError());
        RTP_CUDA_B(cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, kb64, vb, static_cast<int>(n), 0, 64));
        // pass 3 (most significant): the range each item belongs to
        build_segkeys_kernel<<<grid, 256>>>(vb.Current(), d_start, n, kb32.Current());
        RTP_CUDA_B(cudaGetLastError());
        RTP_CUDA_B(cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, kb32, vb, static_cast<int>(n), 0, seg_bits));
        build_split_kernel<<<grid, 256>>>(vb.Current(), n, d_start, d_len);
        RTP_CUDA_B(cudaGetLastError());
    }
    RTP_CUDA_B(cudaMemcpy(d_order_out, vb.Current(), static_cast<size_t>(n) * 4, cudaMemcpyDeviceToDevice));
    cleanup();
    return RTP_OK;
}

}  // namespace rtp

// =================================================================================================================================
// device_build_scene: the rest of the scene build on the GPU (SURVEY.md 8f-1). Everything below restates a host stage of
// rtp_host.cpp with the same arithmetic, so that the trees are equal node for node (tests/test_gpu_parity.py compares digests):
//   leaf boxes             hittable.rs:124-140 (flatten_scene)
//   reference order        bvh.rs:36-67 (above)
//   SAH culling tree       SeqBuilder: split position minimising area(L)|L| + area(R)|R| over the rank-ordered sequence, first minimum
//   records                DPrim / DAttr in rank order (flatten_scene)
//   4-wide collapse        WideBuilder: expand the internal child of largest area until four children
//   any-order tables       prepare_any_order: big primitives (extent > 16 x median, the eight largest), E / A / C / R, scene magnitude
//   order-free tree        prepare_any_order's build_free_tree itself, on the host, over the leaf boxes read back
// The SAH build is level-synchronous: all ranges of one depth are processed by a handful of whole-array passes — a forward and a
// backward segmented scan of box unions (cub::DeviceScan::InclusiveScanByKey: library code for this once-per-scene stage), a cost
// pass with a per-range atomic minimum, and a split pass that writes the nodes of that depth straight into their pre-order slots.
// =================================================================================================================================

#include <cub/device/device_scan.cuh>
#include <math_constants.h>
#include <thrust/iterator/reverse_iterator.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>
#include <vector>

namespace rtp {

struct Box6 {
    double lo[3], hi[3];
};
struct BoxUnion {  // utility.rs:130-135 AABB::union (fmin / fmax: IEEE minNum / maxNum)
    __host__ __device__ Box6 operator()(const Box6& a, const Box6& b) const {
        Box6 r;
        for (int k = 0; k < 3; ++k) { r.lo[k] = fmin(a.lo[k], b.lo[k]); r.hi[k] = fmax(a.hi[k], b.hi[k]); }
        return r;
    }
};
__device__ __forceinline__ double half_area_of(const double* lo, const double* hi) {  // SeqBuilder::Box::half_area, WideBuilder::half_area
    const double dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    const double a = dx * dy + dy * dz + dz * dx;
    return a == a ? a : CUDART_INF;
}

struct MeshRef {  // one rtp_mesh on the device: where its vertices / indices start in the concatenated arrays
    uint64_t vertex_base, index_base;
    uint32_t n_vertices, n_indices, material, _pad;
};

// ---- leaf boxes + validation (flatten_scene "leaf boxes") ----------------------------------------------------------------------------
// status[0]: index << 3 | error class of the smallest failing hittable (all ones: none; one atomic word, so that the class belongs
// to the index), status[1]: 1 = some box is inverted or non-finite
__global__ void __launch_bounds__(256) leaf_boxes_kernel(const rtp_hittable* __restrict__ hs, uint32_t n, const MeshRef* __restrict__ meshes, uint32_t n_meshes,
                                                          uint32_t n_materials, const rtp_vertex* __restrict__ verts, const uint32_t* __restrict__ idx,
                                                          Box6* __restrict__ boxes, unsigned long long* __restrict__ status) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const rtp_hittable h = hs[i];
    Box6 b;
    unsigned int err = 0;
    if (h.kind == RTP_HITTABLE_SPHERE) {
        if (h.material >= n_materials) err = 1;
        for (int k = 0; k < 3; ++k) { b.lo[k] = h.center[k] - h.radius; b.hi[k] = h.center[k] + h.radius; }
    } else if (h.kind == RTP_HITTABLE_TRIANGLE) {
        if (h.mesh >= n_meshes || static_cast<uint64_t>(h.triangle) + 3 > meshes[h.mesh].n_indices) {
            err = 2;
            for (int k = 0; k < 3; ++k) b.lo[k] = b.hi[k] = 0.0;
        } else {
            const MeshRef m = meshes[h.mesh];
            const double* a = verts[m.vertex_base + idx[m.index_base + h.triangle + 0]].position;
            const double* bb = verts[m.vertex_base + idx[m.index_base + h.triangle + 1]].position;
            const double* c = verts[m.vertex_base + idx[m.index_base + h.triangle + 2]].position;
            for (int k = 0; k < 3; ++k) { b.lo[k] = fmin(fmin(a[k], bb[k]), c[k]); b.hi[k] = fmax(fmax(a[k], bb[k]), c[k]); }
        }
    } else {
        err = 3;
        for (int k = 0; k < 3; ++k) b.lo[k] = b.hi[k] = 0.0;
    }
    if (!err)
        for (int k = 0; k < 3; ++k) {
            const double key = 0.5 * (b.lo[k] + b.hi[k]);
            if (key != key) err = 4;  // partial_cmp().unwrap() panics on NaN (bvh.rs:63)
        }
    if (err) atomicMin(&status[0], static_cast<unsigned long long>(i) << 3 | err);
    bool regular = true;
    for (int k = 0; k < 3; ++k)
        if (!(b.lo[k] <= b.hi[k]) || !(fabs(b.lo[k]) <= 1.7976931348623157e308) || !(fabs(b.hi[k]) <= 1.7976931348623157e308)) regular = false;
    if (!regular) status[1] = 1ull;
    boxes[i] = b;
}

__global__ void __launch_bounds__(256) gather_boxes_kernel(const Box6* __restrict__ boxes, const uint32_t* __restrict__ perm, uint32_t n, Box6* __restrict__ ranked) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) ranked[r] = boxes[perm[r]];
}

// ---- SAH over the rank-ordered sequence (SeqBuilder) -----------------------------------------------------------------------------------
struct Seg {
    uint32_t lo, n, base, _pad;  // leaves [lo, lo + n), its node sits at pre-order index `base`
};

constexpr unsigned long long kInfBits = 0x7FF0000000000000ull;

// element i of an active range: cost of cutting AFTER i (left = lo..i), minimised per range; ties go to the smallest position like the
// host's strict `cost < best`
__global__ void __launch_bounds__(256) sah_cost_kernel(const uint32_t* __restrict__ key, const Seg* __restrict__ segs, const Box6* __restrict__ pre, const Box6* __restrict__ suf, uint32_t n,
                                                        unsigned long long* __restrict__ best_cost) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t s = key[i];
    if (s == 0xFFFFFFFFu) return;
    const Seg sg = segs[s];
    if (i + 1u >= sg.lo + sg.n) return;  // the last element of a range is no cut position
    const uint32_t k = i - sg.lo + 1u;
    const double cost = half_area_of(pre[i].lo, pre[i].hi) * static_cast<double>(k) + half_area_of(suf[i + 1].lo, suf[i + 1].hi) * static_cast<double>(sg.n - k);
    atomicMin(&best_cost[s], static_cast<unsigned long long>(__double_as_longlong(cost)));  // costs are >= 0 or +inf: the bit pattern orders like the value
}
__global__ void __launch_bounds__(256) sah_argmin_kernel(const uint32_t* __restrict__ key, const Seg* __restrict__ segs, const Box6* __restrict__ pre, const Box6* __restrict__ suf, uint32_t n,
                                                          const unsigned long long* __restrict__ best_cost, uint32_t* __restrict__ best_k) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t s = key[i];
    if (s == 0xFFFFFFFFu) return;
    const Seg sg = segs[s];
    if (i + 1u >= sg.lo + sg.n) return;
    const uint32_t k = i - sg.lo + 1u;
    const double cost = half_area_of(pre[i].lo, pre[i].hi) * static_cast<double>(k) + half_area_of(suf[i + 1].lo, suf[i + 1].hi) * static_cast<double>(sg.n - k);
    if (static_cast<unsigned long long>(__double_as_longlong(cost)) == best_cost[s]) atomicMin(&best_k[s], k);
}

// one thread per active range: choose the cut, write this range's node and any leaf children, report how many children stay active
__global__ void __launch_bounds__(256) sah_split_kernel(const Seg* __restrict__ segs, uint32_t n_segs, const unsigned long long* __restrict__ best_cost, uint32_t* __restrict__ best_k,
                                                         const Box6* __restrict__ pre, const Box6* __restrict__ ranked, const uint32_t* __restrict__ perm, const rtp_hittable* __restrict__ hs,
                                                         uint32_t level, DNode* __restrict__ nodes, uint32_t* __restrict__ n_active_children) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_segs) return;
    const Seg sg = segs[s];
    // SeqBuilder::build: past 192 levels fall back to the median; choose_split keeps n / 2 when no finite cost exists
    uint32_t k = sg.n / 2;
    if (level < 192u && best_cost[s] < kInfBits) k = best_k[s];
    best_k[s] = k;
    DNode nd;
    const Box6 total = pre[sg.lo + sg.n - 1u];
    for (int a = 0; a < 3; ++a) { nd.bmin[a] = total.lo[a]; nd.bmax[a] = total.hi[a]; }
    nd.skip = sg.base + 2u * sg.n - 1u; nd.prim = kNoPrim; nd.kind = 0; nd._pad = 0;
    nodes[sg.base] = nd;
    uint32_t active = 0;
    const uint32_t child_lo[2] = {sg.lo, sg.lo + k}, child_n[2] = {k, sg.n - k}, child_base[2] = {sg.base + 1u, sg.base + 2u * k};
    for (int c = 0; c < 2; ++c) {
        if (child_n[c] == 1u) {
            DNode lf;
            const Box6 b = ranked[child_lo[c]];
            for (int a = 0; a < 3; ++a) { lf.bmin[a] = b.lo[a]; lf.bmax[a] = b.hi[a]; }
            lf.skip = child_base[c] + 1u; lf.prim = child_lo[c]; lf.kind = hs[perm[child_lo[c]]].kind; lf._pad = 0;
            nodes[child_base[c]] = lf;
        } else {
            ++active;
        }
    }
    n_active_children[s] = active;
}
// second half of the split: the active children become the next level's ranges, at positions given by the exclusive scan of the counts
__global__ void __launch_bounds__(256) sah_emit_kernel(const Seg* __restrict__ segs, uint32_t n_segs, const uint32_t* __restrict__ best_k, const uint32_t* __restrict__ child_pos,
                                                        Seg* __restrict__ next, uint32_t* __restrict__ first_child) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_segs) return;
    const Seg sg = segs[s];
    const uint32_t k = best_k[s];
    uint32_t pos = child_pos[s];
    uint32_t ids[2] = {0xFFFFFFFFu, 0xFFFFFFFFu};
    if (k > 1u) { next[pos] = Seg{sg.lo, k, sg.base + 1u, 0u}; ids[0] = pos++; }
    if (sg.n - k > 1u) { next[pos] = Seg{sg.lo + k, sg.n - k, sg.base + 2u * k, 0u}; ids[1] = pos; }
    first_child[2 * s] = ids[0]; first_child[2 * s + 1] = ids[1];
}
__global__ void __launch_bounds__(256) sah_rekey_kernel(uint32_t* __restrict__ key, const Seg* __restrict__ segs, const uint32_t* __restrict__ best_k, const uint32_t* __restrict__ first_child, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t s = key[i];
    if (s == 0xFFFFFFFFu) return;
    const Seg sg = segs[s];
    key[i] = first_child[2 * s + ((i - sg.lo) >= best_k[s] ? 1 : 0)];  // 0xFFFFFFFF: the element became a leaf
}
__global__ void __launch_bounds__(256) fill_u64_kernel(unsigned long long* p, unsigned long long v, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void __launch_bounds__(256) fill_u32_kernel(uint32_t* p, uint32_t v, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// ---- primitive and attribute records in rank order (flatten_scene "primitives in traversal order") ------------------------------------
__global__ void __launch_bounds__(256) records_kernel(const rtp_hittable* __restrict__ hs, const uint32_t* __restrict__ perm, uint32_t n, const MeshRef* __restrict__ meshes,
                                                       const rtp_vertex* __restrict__ verts, const uint32_t* __restrict__ idx, const Box6* __restrict__ ranked,
                                                       DPrim* __restrict__ prims, DAttr* __restrict__ attrs, double* __restrict__ extent) {
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n) return;
    const uint32_t id = perm[slot];
    const rtp_hittable h = hs[id];
    DPrim p;
    DAttr at;
    memset(&p, 0, sizeof p);
    memset(&at, 0, sizeof at);
    p.leaf = id;
    const Box6 b = ranked[slot];
    for (int k = 0; k < 3; ++k) { p.bmin[k] = b.lo[k]; p.bmax[k] = b.hi[k]; }
    if (h.kind == RTP_HITTABLE_SPHERE) {
        for (int k = 0; k < 3; ++k) p.a[k] = h.center[k];
        p.ba[0] = h.radius;
        p.material = h.material;
    } else {
        const MeshRef m = meshes[h.mesh];
        const rtp_vertex va = verts[m.vertex_base + idx[m.index_base + h.triangle + 0]];
        const rtp_vertex vb = verts[m.vertex_base + idx[m.index_base + h.triangle + 1]];
        const rtp_vertex vc = verts[m.vertex_base + idx[m.index_base + h.triangle + 2]];
        for (int k = 0; k < 3; ++k) {
            p.a[k] = va.position[k];
            p.ba[k] = va.position[k] - vb.position[k];  // hittable.rs:71
            p.ca[k] = va.position[k] - vc.position[k];  // hittable.rs:72
            at.n[0][k] = va.normal[k]; at.n[1][k] = vb.normal[k]; at.n[2][k] = vc.normal[k];
        }
        for (int k = 0; k < 2; ++k) { at.uv[0][k] = va.uv[k]; at.uv[1][k] = vb.uv[k]; at.uv[2][k] = vc.uv[k]; }
        p.material = m.material;  // hittable.rs:107
    }
    prims[slot] = p;
    attrs[slot] = at;
    extent[slot] = fmax(b.hi[0] - b.lo[0], fmax(b.hi[1] - b.lo[1], b.hi[2] - b.lo[2]));  // prepare_any_order: extent()
}

// ---- any-order tables (prepare_any_order) ------------------------------------------------------------------------------------------------
struct AnyConsts {
    unsigned long long E, A, C, R, mag;  // bit patterns of non-negative doubles: atomicMax orders them like the values
    unsigned int spheres, _pad;
    unsigned long long lo[3], hi[3];     // union of the boxes that are not big: ~order_key(min), order_key(max), both by atomicMax
};
// a double's bits as an unsigned key that orders like the value (-0 below +0)
__device__ __forceinline__ unsigned long long order_key(double x) {
    const unsigned long long u = static_cast<unsigned long long>(__double_as_longlong(x));
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
static double from_order_key(unsigned long long k) {
    const unsigned long long u = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
    double x;
    std::memcpy(&x, &u, 8);
    return x;
}
__global__ void __launch_bounds__(256) any_consts_kernel(const DPrim* __restrict__ prims, const rtp_hittable* __restrict__ hs, const double* __restrict__ extent, uint32_t n,
                                                          const uint32_t* __restrict__ big, uint32_t n_big, AnyConsts* __restrict__ out) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const DPrim& p = prims[s];
    double mag = 0.0;
    for (int k = 0; k < 3; ++k) mag = fmax(mag, fmax(fabs(p.bmin[k]), fabs(p.bmax[k])));
    atomicMax(&out->mag, static_cast<unsigned long long>(__double_as_longlong(mag)));
    for (uint32_t k = 0; k < n_big; ++k)
        if ((big[k] & 0x7FFFFFFFu) == s) return;
    for (int k = 0; k < 3; ++k) { atomicMax(&out->lo[k], ~order_key(p.bmin[k])); atomicMax(&out->hi[k], order_key(p.bmax[k])); }
    const bool sphere = hs[p.leaf].kind == RTP_HITTABLE_SPHERE;
    if (sphere) {
        out->spheres = 1u;
        atomicMax(&out->C, static_cast<unsigned long long>(__double_as_longlong(mag)));
        atomicMax(&out->R, static_cast<unsigned long long>(__double_as_longlong(0.5 * extent[s])));
    } else {
        atomicMax(&out->E, static_cast<unsigned long long>(__double_as_longlong(extent[s])));
        atomicMax(&out->A, static_cast<unsigned long long>(__double_as_longlong(mag)));
    }
}
struct Over {
    double ext;
    uint32_t slot, kind;
};
__global__ void __launch_bounds__(256) over_kernel(const double* __restrict__ extent, const DPrim* __restrict__ prims, const rtp_hittable* __restrict__ hs, uint32_t n, double cap,
                                                    Over* __restrict__ out, unsigned int* __restrict__ count, unsigned int max_out) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n || !(extent[s] > cap)) return;
    const unsigned int k = atomicAdd(count, 1u);
    if (k < max_out) out[k] = Over{extent[s], s, hs[prims[s].leaf].kind};
}

// ---- 4-wide collapse (WideBuilder), breadth first: one launch pair per level of the wide tree ------------------------------------------
struct WideTask {
    uint32_t bnode;  // binary node this wide node is collapsed from
};
__device__ __forceinline__ int collapse_kids(const DNode* __restrict__ bn, uint32_t b, uint32_t kids[4]) {
    int nk = 0;
    if (bn[b].prim != kNoPrim) {
        kids[nk++] = b;  // a one-leaf scene: the root holds that leaf as its only child
    } else {
        kids[nk++] = b + 1;
        kids[nk++] = bn[b + 1].skip;
        while (nk < 4) {
            int pick = -1;
            double best = -1.0;
            for (int k = 0; k < nk; ++k)
                if (bn[kids[k]].prim == kNoPrim) {
                    const double a = half_area_of(bn[kids[k]].bmin, bn[kids[k]].bmax);
                    if (a > best) { best = a; pick = k; }
                }
            if (pick < 0) break;
            const uint32_t c = kids[pick];
            for (int k = nk; k > pick + 1; --k) kids[k] = kids[k - 1];
            kids[pick] = c + 1;
            kids[pick + 1] = bn[c + 1].skip;
            ++nk;
        }
    }
    return nk;
}
__global__ void __launch_bounds__(128) collapse_count_kernel(const DNode* __restrict__ bn, const WideTask* __restrict__ tasks, uint32_t m, uint32_t* __restrict__ n_internal) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    uint32_t kids[4];
    const int nk = collapse_kids(bn, tasks[j].bnode, kids);
    uint32_t c = 0;
    for (int k = 0; k < nk; ++k) c += bn[kids[k]].prim == kNoPrim ? 1u : 0u;
    n_internal[j] = c;
}
__device__ __forceinline__ void round_out_dev(const double* bmin, const double* bmax, float* lo, float* hi) {  // rtp_host.cpp round_out
    for (int a = 0; a < 3; ++a) {
        const double mag = fmax(fabs(bmin[a]), fabs(bmax[a]));
        const double r = ldexp(mag, -21);
        float l = static_cast<float>(bmin[a] - r), h = static_cast<float>(bmax[a] + r);
        if (static_cast<double>(l) > bmin[a] - r) l = nextafterf(l, -CUDART_INF_F);
        if (static_cast<double>(h) < bmax[a] + r) h = nextafterf(h, CUDART_INF_F);
        lo[a] = l; hi[a] = h;
    }
}
__global__ void __launch_bounds__(128) collapse_write_kernel(const DNode* __restrict__ bn, const WideTask* __restrict__ tasks, uint32_t m, const uint32_t* __restrict__ child_pos,
                                                              uint32_t level_base, uint32_t next_base, const uint32_t* __restrict__ big, uint32_t n_big,
                                                              DWide* __restrict__ wide, double* __restrict__ wide_boxes, WideTask* __restrict__ next) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    uint32_t kids[4];
    const int nk = collapse_kids(bn, tasks[j].bnode, kids);
    DWide w;
    memset(&w, 0, sizeof w);
    double b64[4][6];
    uint32_t pos = child_pos[j];
    for (int k = 0; k < 4; ++k) {
        if (k < nk) {
            const DNode c = bn[kids[k]];
            float lo[3], hi[3];
            round_out_dev(c.bmin, c.bmax, lo, hi);
            for (int a = 0; a < 3; ++a) { w.plane[a][0][k] = lo[a]; w.plane[a][1][k] = hi[a]; b64[k][a] = c.bmin[a]; b64[k][3 + a] = c.bmax[a]; }
            if (c.prim != kNoPrim) {
                // mark_big: a leaf of one of the big primitives carries kWideBig
                bool is_big = false;
                for (uint32_t q = 0; q < n_big; ++q) is_big |= (big[q] & 0x7FFFFFFFu) == c.prim;
                w.child[k] = kWideLeaf | (c.kind << 30) | c.prim | (is_big ? kWideBig : 0u);
            } else {
                next[pos] = WideTask{kids[k]};
                w.child[k] = next_base + pos;
                ++pos;
            }
        } else {
            for (int a = 0; a < 3; ++a) {
                w.plane[a][0][k] = CUDART_INF_F; w.plane[a][1][k] = -CUDART_INF_F;
                b64[k][a] = CUDART_INF; b64[k][3 + a] = -CUDART_INF;
            }
            w.child[k] = kWideEmpty;
        }
    }
    if (!wide) return;  // sizing sweep: only the next level's tasks are needed
    wide[level_base + j] = w;
    double* dst = wide_boxes + static_cast<size_t>(level_base + j) * 24;
    for (int k = 0; k < 4; ++k)
        for (int a = 0; a < 6; ++a) dst[6 * k + a] = b64[k][a];
}

void device_free_arrays(DevArrays* a) {
    if (!a || !a->valid) return;
    if (a->adopted) { *a = DevArrays{}; return; }  // a DeviceScene owns them
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(a->device);
    cudaFree(a->nodes); cudaFree(a->wide); cudaFree(a->wide_boxes); cudaFree(a->prims); cudaFree(a->attrs);
    if (prev >= 0) cudaSetDevice(prev);
    *a = DevArrays{};
}

int device_build_scene(const rtp_scene_desc* d, const Switches& sw, FlatScene* out) {
    const uint32_t n = d->n_hittables;
    if (n < 2) return 1;
    if (int rc = ensure_device()) return rc;
    auto t0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!sw.build_timing) return;
        cudaDeviceSynchronize();
        auto t1 = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[rtp build, device] %s: %.3f s\n", what, std::chrono::duration<double>(t1 - t0).count());
        t0 = t1;
    };
    std::vector<void*> scratch;  // freed on every exit; the arrays handed to `out->dev` are taken off this list at the end
    auto cleanup = [&]() { for (void* p : scratch) cudaFree(p); scratch.clear(); };
    auto dalloc = [&](void** p, size_t bytes) { cudaError_t e = cudaMalloc(p, bytes ? bytes : 1); if (e == cudaSuccess) scratch.push_back(*p); return e; };
#define RTP_DALLOC(ptr, bytes) RTP_CUDA_B(dalloc(reinterpret_cast<void**>(&(ptr)), (bytes)))

    // ---- inputs: hittables, meshes (vertices and indices concatenated) ---------------------------------------------------------------------
    std::vector<MeshRef> refs(d->n_meshes);
    uint64_t nv = 0, ni = 0;
    for (uint32_t m = 0; m < d->n_meshes; ++m) {
        refs[m] = MeshRef{nv, ni, d->meshes[m].n_vertices, d->meshes[m].n_indices, d->meshes[m].material, 0u};
        nv += d->meshes[m].n_vertices; ni += d->meshes[m].n_indices;
    }
    rtp_hittable* d_hs = nullptr; MeshRef* d_refs = nullptr; rtp_vertex* d_verts = nullptr; uint32_t* d_idx = nullptr;
    RTP_DALLOC(d_hs, static_cast<size_t>(n) * sizeof(rtp_hittable));
    RTP_DALLOC(d_refs, refs.size() * sizeof(MeshRef));
    RTP_DALLOC(d_verts, nv * sizeof(rtp_vertex));
    RTP_DALLOC(d_idx, ni * sizeof(uint32_t));
    RTP_CUDA_B(cudaMemcpy(d_hs, d->hittables, static_cast<size_t>(n) * sizeof(rtp_hittable), cudaMemcpyHostToDevice));
    if (!refs.empty()) RTP_CUDA_B(cudaMemcpy(d_refs, refs.data(), refs.size() * sizeof(MeshRef), cudaMemcpyHostToDevice));
    for (uint32_t m = 0; m < d->n_meshes; ++m) {
        if (refs[m].n_vertices) RTP_CUDA_B(cudaMemcpy(d_verts + refs[m].vertex_base, d->meshes[m].vertices, static_cast<size_t>(refs[m].n_vertices) * sizeof(rtp_vertex), cudaMemcpyHostToDevice));
        if (refs[m].n_indices) RTP_CUDA_B(cudaMemcpy(d_idx + refs[m].index_base, d->meshes[m].indices, static_cast<size_t>(refs[m].n_indices) * sizeof(uint32_t), cudaMemcpyHostToDevice));
    }
    lap("inputs to the device (hittables, vertices, indices)");

    // ---- leaf boxes + validation -----------------------------------------------------------------------------------------------------------
    const unsigned grid = (n + 255) / 256;
    Box6 *d_boxes = nullptr, *d_ranked = nullptr;
    unsigned long long* d_status = nullptr;
    RTP_DALLOC(d_boxes, static_cast<size_t>(n) * sizeof(Box6));
    RTP_DALLOC(d_ranked, static_cast<size_t>(n) * sizeof(Box6));
    RTP_DALLOC(d_status, 2 * sizeof(unsigned long long));
    {
        const unsigned long long init[2] = {~0ull, 0ull};
        RTP_CUDA_B(cudaMemcpy(d_status, init, sizeof init, cudaMemcpyHostToDevice));
    }
    leaf_boxes_kernel<<<grid, 256>>>(d_hs, n, d_refs, d->n_meshes, d->n_materials, d_verts, d_idx, d_boxes, d_status);
    RTP_CUDA_B(cudaGetLastError());
    unsigned long long status[2];
    RTP_CUDA_B(cudaMemcpy(status, d_status, sizeof status, cudaMemcpyDeviceToHost));
    if (status[0] != ~0ull) {
        cleanup();
        const uint64_t bad = status[0] >> 3;
        switch (status[0] & 7u) {
            case 1: return set_error(RTP_ERR_INVALID, "sphere material out of range");
            case 2: return set_error(RTP_ERR_INVALID, "triangle id out of range");
            case 4: return set_error(RTP_ERR_INVALID, "NaN bounding-box centroid in hittable " + std::to_string(bad));
            default: return set_error(RTP_ERR_INVALID, "unknown hittable kind");
        }
    }
    if (status[1]) { cleanup(); return 1; }  // inverted / non-finite boxes keep the reference topology: host path (DESIGN.md §2)
    lap("leaf boxes and validation");

    // ---- reference order (bvh.rs:36-67), boxes stay on the device ----------------------------------------------------------------------------
    uint32_t* d_perm = nullptr;
    RTP_DALLOC(d_perm, static_cast<size_t>(n) * sizeof(uint32_t));
    {
        int rc = device_reference_order_dev(reinterpret_cast<const double*>(d_boxes), n, d_perm);
        if (rc != RTP_OK) { cleanup(); return rc; }
    }
    gather_boxes_kernel<<<grid, 256>>>(d_boxes, d_perm, n, d_ranked);
    RTP_CUDA_B(cudaGetLastError());
    out->leaf_order.resize(n);
    RTP_CUDA_B(cudaMemcpy(out->leaf_order.data(), d_perm, static_cast<size_t>(n) * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    lap("reference order (segmented radix sorts)");

    // ---- SAH culling tree over the rank order, level by level -----------------------------------------------------------------------------------
    DNode* d_nodes = nullptr;
    const size_t n_nodes = static_cast<size_t>(2) * n - 1;
    RTP_DALLOC(d_nodes, n_nodes * sizeof(DNode));
    Box6 *d_pre = nullptr, *d_suf = nullptr;
    uint32_t *d_key = nullptr, *d_best_k = nullptr, *d_cnt = nullptr, *d_pos = nullptr, *d_first = nullptr;
    unsigned long long* d_best_cost = nullptr;
    Seg* d_segs[2] = {nullptr, nullptr};
    const uint32_t max_segs = n / 2 + 1;
    RTP_DALLOC(d_pre, static_cast<size_t>(n) * sizeof(Box6));
    RTP_DALLOC(d_suf, static_cast<size_t>(n) * sizeof(Box6));
    RTP_DALLOC(d_key, static_cast<size_t>(n) * 4);
    RTP_DALLOC(d_best_k, static_cast<size_t>(max_segs) * 4);
    RTP_DALLOC(d_cnt, static_cast<size_t>(max_segs) * 4);
    RTP_DALLOC(d_pos, static_cast<size_t>(max_segs) * 4);
    RTP_DALLOC(d_first, static_cast<size_t>(max_segs) * 8);
    RTP_DALLOC(d_best_cost, static_cast<size_t>(max_segs) * 8);
    RTP_DALLOC(d_segs[0], static_cast<size_t>(max_segs) * sizeof(Seg));
    RTP_DALLOC(d_segs[1], static_cast<size_t>(max_segs) * sizeof(Seg));
    size_t temp_bytes = 0, need = 0;
    void* d_temp = nullptr;
    {
        auto rkey = thrust::make_reverse_iterator(d_key + n);
        auto rin = thrust::make_reverse_iterator(d_ranked + n);
        auto rout = thrust::make_reverse_iterator(d_suf + n);
        RTP_CUDA_B(cub::DeviceScan::InclusiveScanByKey(nullptr, need, d_key, d_ranked, d_pre, BoxUnion(), static_cast<int>(n)));
        temp_bytes = need;
        RTP_CUDA_B(cub::DeviceScan::InclusiveScanByKey(nullptr, need, rkey, rin, rout, BoxUnion(), static_cast<int>(n)));
        temp_bytes = std::max(temp_bytes, need);
        RTP_CUDA_B(cub::DeviceScan::ExclusiveSum(nullptr, need, d_cnt, d_pos, static_cast<int>(max_segs)));
        temp_bytes = std::max(temp_bytes, need);
        RTP_DALLOC(d_temp, temp_bytes);
    }
    {
        const Seg root{0u, n, 0u, 0u};
        RTP_CUDA_B(cudaMemcpy(d_segs[0], &root, sizeof root, cudaMemcpyHostToDevice));
        RTP_CUDA_B(cudaMemset(d_key, 0, static_cast<size_t>(n) * 4));
    }
    uint32_t n_segs = 1, level = 1, sah_depth = 1;
    int cur = 0;
    while (n_segs > 0) {
        auto rkey = thrust::make_reverse_iterator(d_key + n);
        auto rin = thrust::make_reverse_iterator(d_ranked + n);
        auto rout = thrust::make_reverse_iterator(d_suf + n);
        RTP_CUDA_B(cub::DeviceScan::InclusiveScanByKey(d_temp, temp_bytes, d_key, d_ranked, d_pre, BoxUnion(), static_cast<int>(n)));
        RTP_CUDA_B(cub::DeviceScan::InclusiveScanByKey(d_temp, temp_bytes, rkey, rin, rout, BoxUnion(), static_cast<int>(n)));
        const unsigned sgrid = (n_segs + 255) / 256;
        fill_u64_kernel<<<sgrid, 256>>>(d_best_cost, 0xFFFFFFFFFFFFFFFFull, n_segs);
        fill_u32_kernel<<<sgrid, 256>>>(d_best_k, 0xFFFFFFFFu, n_segs);
        sah_cost_kernel<<<grid, 256>>>(d_key, d_segs[cur], d_pre, d_suf, n, d_best_cost);
        sah_argmin_kernel<<<grid, 256>>>(d_key, d_segs[cur], d_pre, d_suf, n, d_best_cost, d_best_k);
        sah_split_kernel<<<sgrid, 256>>>(d_segs[cur], n_segs, d_best_cost, d_best_k, d_pre, d_ranked, d_perm, d_hs, level, d_nodes, d_cnt);
        RTP_CUDA_B(cudaGetLastError());
        RTP_CUDA_B(cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, d_cnt, d_pos, static_cast<int>(n_segs)));
        sah_emit_kernel<<<sgrid, 256>>>(d_segs[cur], n_segs, d_best_k, d_pos, d_segs[cur ^ 1], d_first);
        sah_rekey_kernel<<<grid, 256>>>(d_key, d_segs[cur], d_best_k, d_first, n);
        RTP_CUDA_B(cudaGetLastError());
        uint32_t last_pos = 0, last_cnt = 0;
        RTP_CUDA_B(cudaMemcpy(&last_pos, d_pos + (n_segs - 1), 4, cudaMemcpyDeviceToHost));
        RTP_CUDA_B(cudaMemcpy(&last_cnt, d_cnt + (n_segs - 1), 4, cudaMemcpyDeviceToHost));
        n_segs = last_pos + last_cnt;
        cur ^= 1;
        ++level;
        sah_depth = level;  // the children of this level's ranges sit one level below
    }
    out->device_depth = sah_depth;
    lap("SAH culling tree over the rank order (level-synchronous)");

    // ---- primitive / attribute records -----------------------------------------------------------------------------------------------------------
    DPrim* d_prims = nullptr; DAttr* d_attrs = nullptr; double* d_ext = nullptr;
    RTP_DALLOC(d_prims, static_cast<size_t>(n) * sizeof(DPrim));
    RTP_DALLOC(d_attrs, static_cast<size_t>(n) * sizeof(DAttr));
    RTP_DALLOC(d_ext, static_cast<size_t>(n) * sizeof(double));
    records_kernel<<<grid, 256>>>(d_hs, d_perm, n, d_refs, d_verts, d_idx, d_ranked, d_prims, d_attrs, d_ext);
    RTP_CUDA_B(cudaGetLastError());
    lap("primitive and attribute records");

    // ---- any-order tables: big primitives, slack constants, scene magnitude (prepare_any_order) --------------------------------------------------
    uint32_t h_big[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t n_big = 0;
    {
        // median extent: element n / 2 of the sorted extents (std::nth_element's answer); extents are >= 0, so their bit patterns sort like the values
        double *d_sorted = nullptr, *d_keys_in = nullptr;
        RTP_DALLOC(d_sorted, static_cast<size_t>(n) * 8);
        RTP_DALLOC(d_keys_in, static_cast<size_t>(n) * 8);
        RTP_CUDA_B(cudaMemcpy(d_keys_in, d_ext, static_cast<size_t>(n) * 8, cudaMemcpyDeviceToDevice));
        size_t sb = 0;
        RTP_CUDA_B(cub::DeviceRadixSort::SortKeys(nullptr, sb, reinterpret_cast<unsigned long long*>(d_keys_in), reinterpret_cast<unsigned long long*>(d_sorted), static_cast<int>(n)));
        void* d_st = nullptr;
        RTP_DALLOC(d_st, sb);
        RTP_CUDA_B(cub::DeviceRadixSort::SortKeys(d_st, sb, reinterpret_cast<unsigned long long*>(d_keys_in), reinterpret_cast<unsigned long long*>(d_sorted), static_cast<int>(n)));
        double median = 0.0;
        RTP_CUDA_B(cudaMemcpy(&median, d_sorted + n / 2, 8, cudaMemcpyDeviceToHost));
        const double cap = 16.0 * median;
        const unsigned int max_over = 1u << 20;
        Over* d_over = nullptr; unsigned int* d_count = nullptr;
        RTP_DALLOC(d_over, static_cast<size_t>(max_over) * sizeof(Over));
        RTP_DALLOC(d_count, 4);
        RTP_CUDA_B(cudaMemset(d_count, 0, 4));
        over_kernel<<<grid, 256>>>(d_ext, d_prims, d_hs, n, cap, d_over, d_count, max_over);
        RTP_CUDA_B(cudaGetLastError());
        unsigned int count = 0;
        RTP_CUDA_B(cudaMemcpy(&count, d_count, 4, cudaMemcpyDeviceToHost));
        if (count > max_over) { cleanup(); return 1; }  // a scene where over a million primitives are outsized: leave it to the host path
        std::vector<Over> over(count);
        if (count) RTP_CUDA_B(cudaMemcpy(over.data(), d_over, static_cast<size_t>(count) * sizeof(Over), cudaMemcpyDeviceToHost));
        std::sort(over.begin(), over.end(), [](const Over& a, const Over& b) { return a.ext != b.ext ? a.ext > b.ext : a.slot < b.slot; });
        for (size_t k = 0; k < over.size() && n_big < kMaxBig; ++k) h_big[n_big++] = over[k].slot | (over[k].kind << 31);
    }
    uint32_t* d_big = nullptr;
    AnyConsts* d_consts = nullptr;
    RTP_DALLOC(d_big, sizeof h_big);
    RTP_DALLOC(d_consts, sizeof(AnyConsts));
    RTP_CUDA_B(cudaMemcpy(d_big, h_big, sizeof h_big, cudaMemcpyHostToDevice));
    RTP_CUDA_B(cudaMemset(d_consts, 0, sizeof(AnyConsts)));
    any_consts_kernel<<<grid, 256>>>(d_prims, d_hs, d_ext, n, d_big, n_big, d_consts);
    RTP_CUDA_B(cudaGetLastError());
    AnyConsts hc;
    RTP_CUDA_B(cudaMemcpy(&hc, d_consts, sizeof hc, cudaMemcpyDeviceToHost));
    auto as_double = [](unsigned long long u) { double x; std::memcpy(&x, &u, 8); return x; };
    lap("any-order tables");

    // ---- 4-wide collapse, breadth first: a counting sweep sizes the arrays, a writing sweep fills them ------------------------------------------
    WideTask* d_tasks[2] = {nullptr, nullptr};
    uint32_t *d_wcnt = nullptr, *d_wpos = nullptr;
    RTP_DALLOC(d_tasks[0], static_cast<size_t>(n) * sizeof(WideTask));
    RTP_DALLOC(d_tasks[1], static_cast<size_t>(n) * sizeof(WideTask));
    RTP_DALLOC(d_wcnt, static_cast<size_t>(n) * 4);
    RTP_DALLOC(d_wpos, static_cast<size_t>(n) * 4);
    size_t wtemp = 0;
    RTP_CUDA_B(cub::DeviceScan::ExclusiveSum(nullptr, wtemp, d_wcnt, d_wpos, static_cast<int>(n)));
    void* d_wtemp = nullptr;
    RTP_DALLOC(d_wtemp, wtemp);
    std::vector<uint32_t> level_size;
    DWide* d_wide = nullptr; double* d_wboxes = nullptr;
    size_t n_wide = 0;
    for (int pass = 0; pass < 2; ++pass) {
        if (pass == 1) {
            // as prepare_any_order: a tree too deep for the any-order walk's stack gets no any-order tables, so no leaf is marked big
            if (level_size.size() > 48) { n_big = 0; std::fill(h_big, h_big + 8, 0u); }
            for (uint32_t m : level_size) n_wide += m;
            RTP_DALLOC(d_wide, n_wide * sizeof(DWide));
            RTP_DALLOC(d_wboxes, n_wide * 24 * sizeof(double));
        }
        const WideTask root{0u};
        RTP_CUDA_B(cudaMemcpy(d_tasks[0], &root, sizeof root, cudaMemcpyHostToDevice));
        uint32_t m = 1, base = 0;
        int c = 0;
        for (size_t lv = 0; m > 0; ++lv) {
            const unsigned wgrid = (m + 127) / 128;
            collapse_count_kernel<<<wgrid, 128>>>(d_nodes, d_tasks[c], m, d_wcnt);
            RTP_CUDA_B(cudaGetLastError());
            RTP_CUDA_B(cub::DeviceScan::ExclusiveSum(d_wtemp, wtemp, d_wcnt, d_wpos, static_cast<int>(m)));
            uint32_t last_pos = 0, last_cnt = 0;
            RTP_CUDA_B(cudaMemcpy(&last_pos, d_wpos + (m - 1), 4, cudaMemcpyDeviceToHost));
            RTP_CUDA_B(cudaMemcpy(&last_cnt, d_wcnt + (m - 1), 4, cudaMemcpyDeviceToHost));
            const uint32_t next_m = last_pos + last_cnt;
            if (pass == 0) level_size.push_back(m);
            // the writing kernel also emits the next level's tasks; the counting pass needs them too, so it runs in both passes with
            // pass 0 writing into throw-away rows (skipped: pass 0 only needs the tasks)
            if (pass == 1) {
                collapse_write_kernel<<<wgrid, 128>>>(d_nodes, d_tasks[c], m, d_wpos, base, base + m, d_big, n_big, d_wide, d_wboxes, d_tasks[c ^ 1]);
            } else {
                collapse_write_kernel<<<wgrid, 128>>>(d_nodes, d_tasks[c], m, d_wpos, 0u, 0u, d_big, n_big, nullptr, nullptr, d_tasks[c ^ 1]);
            }
            RTP_CUDA_B(cudaGetLastError());
            base += m;
            m = next_m;
            c ^= 1;
        }
    }
    lap("4-wide collapse (breadth first)");

    // ---- order-free culling tree: the host's builder over the leaf boxes, read back ----------------------------------------------------------
    const bool any_ok = level_size.size() <= 48;
    out->n_big = n_big;
    if (any_ok && n > n_big && want_free_tree(sw, n)) {
        std::vector<Box6> boxes(n);
        RTP_CUDA_B(cudaMemcpy(boxes.data(), d_ranked, static_cast<size_t>(n) * sizeof(Box6), cudaMemcpyDeviceToHost));
        std::vector<uint8_t> kind(n), is_big(n, 0);
        for (uint32_t s = 0; s < n; ++s) kind[s] = static_cast<uint8_t>(d->hittables[out->leaf_order[s]].kind);
        for (uint32_t k = 0; k < n_big; ++k) is_big[h_big[k] & 0x7FFFFFFFu] = 1;
        build_free_tree(boxes[0].lo, boxes[0].hi, sizeof(Box6) / sizeof(double), kind, is_big, out);
        lap("order-free culling tree (host)");
    }

    // ---- hand over -------------------------------------------------------------------------------------------------------------------------------
    RTP_CUDA_B(cudaDeviceSynchronize());
    auto keep = [&](void* p) { scratch.erase(std::remove(scratch.begin(), scratch.end(), p), scratch.end()); };
    keep(d_nodes); keep(d_wide); keep(d_wboxes); keep(d_prims); keep(d_attrs);
    cleanup();
    int device = 0;
    cudaGetDevice(&device);
    out->dev.valid = true; out->dev.device = device;
    out->dev.nodes = d_nodes; out->dev.n_nodes = n_nodes;
    out->dev.wide = d_wide; out->dev.wide_boxes = d_wboxes; out->dev.n_wide = n_wide;
    out->dev.prims = d_prims; out->dev.attrs = d_attrs; out->dev.n_prims = n;
    out->wide_depth = static_cast<uint32_t>(level_size.size());
    out->n_reference_nodes = static_cast<uint32_t>(n_nodes);
    {   // depth of the reference's median-split tree (bvh.rs:36-56): the right half of a range is never smaller than the left
        uint32_t depth = 1;
        for (uint64_t len = n; len > 1; len = len - len / 2) ++depth;
        out->depth = depth;
    }
    out->boxes_finite = true;
    out->scene_mag = as_double(hc.mag);
    out->any_ok = any_ok;
    if (any_ok) {
        for (int k = 0; k < 8; ++k) out->big[k] = h_big[k];
        out->any_E = as_double(hc.E) * (1.0 + 1e-12);
        out->any_A = as_double(hc.A) * (1.0 + 1e-12);
        out->any_C = as_double(hc.C) * (1.0 + 1e-12);
        out->any_R = as_double(hc.R) * (1.0 + 1e-12);
        out->any_spheres = hc.spheres != 0u;
        double lo[3], hi[3];
        for (int k = 0; k < 3; ++k) { lo[k] = from_order_key(~hc.lo[k]); hi[k] = from_order_key(hc.hi[k]); }
        if (hc.hi[0] == 0ull) lo[0] = 1.0, hi[0] = 0.0;  // every primitive is big: the empty box
        culled_set_box(lo, hi, out->cull);
    }
    return RTP_OK;
#undef RTP_DALLOC
}

}  // namespace rtp

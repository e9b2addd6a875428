// rtp_host.cpp — host layer behind the C ABI: error plumbing, asset readers, the reference's
// BVH construction and the flattening of a scene description into the device layout.
//
// Everything here runs once per scene (or per file); none of it is on the per-ray path.
// Reference citations are file:line under /root/reference/src.

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <future>
#include <limits>
#include <mutex>
#include <sstream>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "rtp_internal.h"

namespace rtp {

static thread_local std::string g_last_error;

int set_error(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

// The only reader of the environment (Switches, rtp_internal.h). `unset` is the value of a switch that is not set.
static const char* env(const char* name) { return std::getenv(name); }
static int env_flag(const char* name, int unset) {
    const char* v = env(name);
    return v ? (std::atoi(v) != 0 ? 1 : 0) : unset;
}
static long long env_number(const char* name, long long unset, long long lo, long long hi) {
    const char* v = env(name);
    return v ? std::min(hi, std::max(lo, std::atoll(v))) : unset;
}
static bool env_word(const char* name, const char* word) {
    const char* v = env(name);
    return v && std::strcmp(v, word) == 0;
}

Switches read_switches() {
    Switches s;
    s.any_order = !env_word("RTP_TRAVERSAL", "inorder");
    s.f32_culling = env_flag("RTP_F32_CULLING", s.f32_culling);
    s.simple_trace = env_word("RTP_TRACE_KERNEL", "simple");
    s.simple_render = env_word("RTP_RENDER_KERNEL", "simple");
    s.reference_tree = env_word("RTP_TREE", "reference");
    s.free_tree = env_flag("RTP_FREE_TREE", s.free_tree);
    s.device_build = env_flag("RTP_DEVICE_BUILD", s.device_build);
    s.any_cap = static_cast<uint32_t>(env_number("RTP_ANY_CAP", s.any_cap, 4, 48));
    s.any_setup_cull = env_flag("RTP_ANY_SETUP_CULL", s.any_setup_cull);
    s.tail_threshold = static_cast<uint32_t>(env_number("RTP_TAIL_THRESHOLD", s.tail_threshold, 0, std::numeric_limits<uint32_t>::max()));
    s.chunk_log2 = static_cast<uint32_t>(env_number("RTP_CHUNK_LOG2", s.chunk_log2, 10, 24));
    s.build_timing = env_flag("RTP_BUILD_TIMING", s.build_timing);
    s.debug_sync = env_flag("RTP_DEBUG_SYNC", s.debug_sync);
    s.lane_stats = env_flag("RTP_LANE_STATS", s.lane_stats);
    return s;
}

size_t read_path_budget() { return static_cast<size_t>(env_number("RTP_PATH_BUDGET", 0, 1, 1ll << 31)); }

// f64::min / f64::max (IEEE minNum / maxNum), as used by AABB::union and the triangle box.
static inline double min_num(double a, double b) { return std::fmin(a, b); }
static inline double max_num(double a, double b) { return std::fmax(a, b); }

// nalgebra 0.29 reductions on static 3-vectors: (x*x' + y*y') + z*z'
static inline double dot3(const double* a, const double* b) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; }

// Runs fn(begin, end) over [0, n) in contiguous chunks on the host cores (scene flattening of multi-million-leaf scenes).
template <class F>
static void parallel_chunks(size_t n, F fn) {
    const size_t hw = std::max<size_t>(1, std::min<size_t>(std::thread::hardware_concurrency(), 32));
    const size_t workers = n < 262144 ? 1 : hw;
    if (workers == 1) { fn(size_t(0), n); return; }
    std::vector<std::thread> pool;
    const size_t per = (n + workers - 1) / workers;
    for (size_t w = 0; w < workers; ++w) {
        const size_t b = w * per, e = std::min(n, b + per);
        if (b >= e) break;
        pool.emplace_back([=] { fn(b, e); });
    }
    for (std::thread& t : pool) t.join();
}

// --------------------------------------------------------------------------- BVH build --------

struct BuildItem {
    uint32_t id;  // LeafId
    double bmin[3], bmax[3];
};

struct Builder {
    std::vector<BuildItem>& items;
    std::vector<DNode>& nodes;
    std::atomic<uint32_t> depth{0};

    // bvh.rs:36-56 make_bvh + bvh.rs:58-67 split, writing nodes straight into pre-order position.
    // A range of n leaves occupies 2n-1 consecutive nodes starting at `base`; the left half
    // [lo, lo+n/2) comes first. The reference sorts with sort_unstable_by, whose order among equal
    // centroid keys is unspecified (it depends on the Rust std version); ties are broken by
    // LeafId here, which makes the key a total order and the tree unique.
    void build(size_t lo, size_t n, uint32_t base, int axis, uint32_t level, int spawn_levels) {
        uint32_t seen = depth.load(std::memory_order_relaxed);
        while (level > seen && !depth.compare_exchange_weak(seen, level, std::memory_order_relaxed)) {}
        DNode& nd = nodes[base];
        nd.skip = base + static_cast<uint32_t>(2 * n - 1);
        nd._pad = 0;
        if (n == 1) {
            const BuildItem& it = items[lo];
            std::memcpy(nd.bmin, it.bmin, sizeof nd.bmin);
            std::memcpy(nd.bmax, it.bmax, sizeof nd.bmax);
            nd.prim = static_cast<uint32_t>(lo);
            nd.kind = 0;  // filled by the caller once primitives are laid out
            return;
        }
        std::sort(items.begin() + lo, items.begin() + lo + n, [axis](const BuildItem& x, const BuildItem& y) {
            double kx = 0.5 * (x.bmin[axis] + x.bmax[axis]);
            double ky = 0.5 * (y.bmin[axis] + y.bmax[axis]);
            if (kx != ky) return kx < ky;
            return x.id < y.id;
        });
        size_t nl = n / 2, nr = n - nl;
        uint32_t left = base + 1, right = base + 1 + static_cast<uint32_t>(2 * nl - 1);
        int next_axis = (axis + 1) % 3;
        if (spawn_levels > 0 && n > 65536) {
            auto fut = std::async(std::launch::async, [this, lo, nl, left, next_axis, level, spawn_levels] { build(lo, nl, left, next_axis, level + 1, spawn_levels - 1); });
            build(lo + nl, nr, right, next_axis, level + 1, spawn_levels - 1);
            fut.get();
        } else {
            build(lo, nl, left, next_axis, level + 1, 0);
            build(lo + nl, nr, right, next_axis, level + 1, 0);
        }
        const DNode& l = nodes[left];
        const DNode& r = nodes[right];
        for (int k = 0; k < 3; ++k) {  // utility.rs:130-135 AABB::union
            nd.bmin[k] = min_num(l.bmin[k], r.bmin[k]);
            nd.bmax[k] = max_num(l.bmax[k], r.bmax[k]);
        }
        nd.prim = kNoPrim;
        nd.kind = 0;
    }
};

// ---------------------------------------------------------------------------------------------
// Device culling tree. The reference tree above fixes the ORDER in which leaves are met (its
// depth-first rank) and nothing else: `Bvh::hit` is equivalent to scanning the leaves in rank
// order, testing each leaf's own box and then its primitive against the running t_max, because an
// ancestor box is a superset of the leaf box and IEEE rounding is monotone, so an ancestor test can
// never reject a leaf whose own gate would pass (DESIGN.md §2). Any binary tree over the
// rank-ordered leaf sequence therefore yields identical results, and we are free to choose the
// split positions by surface-area heuristic instead of the median. (With the ground sphere of the
// bunny scenes the median tree drags a 2000-unit box down 13 levels; the SAH tree isolates it.)
// ---------------------------------------------------------------------------------------------
struct SeqBuilder {
    const std::vector<BuildItem>& items;  // in rank order
    std::vector<DNode>& nodes;            // pre-order output, 2n-1 entries
    std::atomic<uint32_t> depth{0};

    struct Box {
        double lo[3], hi[3];
        void reset() { for (int k = 0; k < 3; ++k) { lo[k] = std::numeric_limits<double>::infinity(); hi[k] = -lo[k]; } }
        void grow(const double* bmin, const double* bmax) {
            for (int k = 0; k < 3; ++k) { lo[k] = std::fmin(lo[k], bmin[k]); hi[k] = std::fmax(hi[k], bmax[k]); }
        }
        double half_area() const {
            const double dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
            const double a = dx * dy + dy * dz + dz * dx;
            return a == a ? a : std::numeric_limits<double>::infinity();
        }
    };

    // split position k in [1, n-1] minimising area(L)*|L| + area(R)*|R|, the FIRST minimum (strict <); no finite cost: n / 2.
    // One backward sweep for the suffix areas, one forward sweep for the costs: O(n) per range, O(n log n) per tree. The device
    // build (rtp_build.cu sah_cost_kernel) evaluates the same expression at every position, so both trees are equal node for node.
    size_t choose_split(size_t lo, size_t n) const {
        thread_local std::vector<double> suffix;
        suffix.assign(n + 1, 0.0);
        Box b;
        b.reset();
        for (size_t g = n; g-- > 1;) {  // suffix[g] = area of leaves g..n-1
            b.grow(items[lo + g].bmin, items[lo + g].bmax);
            suffix[g] = b.half_area();
        }
        b.reset();
        double best = std::numeric_limits<double>::infinity();
        size_t best_k = n / 2;
        for (size_t g = 0; g + 1 < n; ++g) {
            b.grow(items[lo + g].bmin, items[lo + g].bmax);
            const size_t k = g + 1;
            const double cost = b.half_area() * static_cast<double>(k) + suffix[k] * static_cast<double>(n - k);
            if (cost < best) { best = cost; best_k = k; }
        }
        return best_k;
    }

    void build(size_t lo, size_t n, uint32_t base, uint32_t level, int spawn_levels) {
        uint32_t seen = depth.load(std::memory_order_relaxed);
        while (level > seen && !depth.compare_exchange_weak(seen, level, std::memory_order_relaxed)) {}
        DNode& nd = nodes[base];
        nd.skip = base + static_cast<uint32_t>(2 * n - 1);
        nd._pad = 0;
        nd.kind = 0;
        if (n == 1) {
            std::memcpy(nd.bmin, items[lo].bmin, sizeof nd.bmin);
            std::memcpy(nd.bmax, items[lo].bmax, sizeof nd.bmax);
            nd.prim = static_cast<uint32_t>(lo);
            return;
        }
        // a pathological chain cannot exhaust the host stack: past 192 levels fall back to the median
        const size_t nl = level < 192 ? choose_split(lo, n) : n / 2, nr = n - nl;
        const uint32_t left = base + 1, right = base + 1 + static_cast<uint32_t>(2 * nl - 1);
        if (spawn_levels > 0 && n > 65536) {
            auto fut = std::async(std::launch::async, [this, lo, nl, left, level, spawn_levels] { build(lo, nl, left, level + 1, spawn_levels - 1); });
            build(lo + nl, nr, right, level + 1, spawn_levels - 1);
            fut.get();
        } else {
            build(lo, nl, left, level + 1, 0);
            build(lo + nl, nr, right, level + 1, 0);
        }
        const DNode& l = nodes[left];
        const DNode& r = nodes[right];
        for (int k = 0; k < 3; ++k) {
            nd.bmin[k] = min_num(l.bmin[k], r.bmin[k]);
            nd.bmax[k] = max_num(l.bmax[k], r.bmax[k]);
        }
        nd.prim = kNoPrim;
    }
};

// ---------------------------------------------------------------------------------------------
// 4-wide f32 culling tree (rtp_internal.h DWide), collapsed from the binary pre-order tree in `nodes`: a node starts with
// its two binary children and repeatedly replaces the internal child of largest surface area by that child's two
// children, in place, until it has four children or only leaves. In-place replacement keeps the children in rank order,
// so visiting children left to right meets the leaves in the reference's depth-first order.
// ---------------------------------------------------------------------------------------------
void round_out(const double* bmin, const double* bmax, float* lo, float* hi) {
    for (int a = 0; a < 3; ++a) {
        const double mag = std::fmax(std::fabs(bmin[a]), std::fabs(bmax[a]));
        const double r = std::ldexp(mag, -21);
        float l = static_cast<float>(bmin[a] - r), h = static_cast<float>(bmax[a] + r);
        if (static_cast<double>(l) > bmin[a] - r) l = std::nextafterf(l, -std::numeric_limits<float>::infinity());
        if (static_cast<double>(h) < bmax[a] + r) h = std::nextafterf(h, std::numeric_limits<float>::infinity());
        lo[a] = l; hi[a] = h;
    }
}

void culled_set_box(const double* lo, const double* hi, float* cull) {
    if (!(lo[0] <= hi[0])) {
        for (int a = 0; a < 3; ++a) { cull[a] = std::numeric_limits<float>::infinity(); cull[3 + a] = -std::numeric_limits<float>::infinity(); }
        return;
    }
    round_out(lo, hi, cull, cull + 3);
}

struct WideBuilder {
    const std::vector<DNode>& bn;
    size_t defer_leaves = 0;  // > 0: subtrees of at most this many leaves are recorded in `deferred` instead of being built
    std::vector<DWide> wide;
    std::vector<double> boxes;  // 24 doubles per wide node: the exact f64 child boxes
    uint32_t depth = 0;
    struct Deferred { uint32_t bnode, parent, slot, depth; };
    std::vector<Deferred> deferred;

    double half_area(uint32_t b) const {
        const double dx = bn[b].bmax[0] - bn[b].bmin[0], dy = bn[b].bmax[1] - bn[b].bmin[1], dz = bn[b].bmax[2] - bn[b].bmin[2];
        const double a = dx * dy + dy * dz + dz * dx;
        return a == a ? a : std::numeric_limits<double>::infinity();
    }

    // builds the subtree under binary node `root_b` into wide[0..), root at index 0
    void run(uint32_t root_b, uint32_t depth0) {
        struct Todo { uint32_t bnode, wnode, depth; };
        std::vector<Todo> todo;
        wide.emplace_back();
        todo.push_back({root_b, 0u, depth0});
        while (!todo.empty()) {
            const Todo t = todo.back();
            todo.pop_back();
            depth = std::max(depth, t.depth);
            uint32_t kids[4];
            int nk = 0;
            if (bn[t.bnode].prim != kNoPrim) {
                kids[nk++] = t.bnode;  // a one-leaf scene: the root holds that leaf as its only child
            } else {
                kids[nk++] = t.bnode + 1;
                kids[nk++] = bn[t.bnode + 1].skip;
                while (nk < 4) {
                    int pick = -1;
                    double best = -1.0;
                    for (int k = 0; k < nk; ++k)
                        if (bn[kids[k]].prim == kNoPrim) {
                            const double a = half_area(kids[k]);
                            if (a > best) { best = a; pick = k; }
                        }
                    if (pick < 0) break;
                    const uint32_t b = kids[pick];
                    for (int k = nk; k > pick + 1; --k) kids[k] = kids[k - 1];
                    kids[pick] = b + 1;
                    kids[pick + 1] = bn[b + 1].skip;
                    ++nk;
                }
            }
            DWide w;
            std::memset(&w, 0, sizeof w);
            double b64[4][6];
            for (int k = 0; k < 4; ++k) {
                if (k < nk) {
                    const DNode& c = bn[kids[k]];
                    float lo[3], hi[3];
                    round_out(c.bmin, c.bmax, lo, hi);
                    for (int a = 0; a < 3; ++a) { w.plane[a][0][k] = lo[a]; w.plane[a][1][k] = hi[a]; b64[k][a] = c.bmin[a]; b64[k][3 + a] = c.bmax[a]; }
                    if (c.prim != kNoPrim) {
                        w.child[k] = kWideLeaf | (c.kind << 30) | c.prim;
                    } else if (defer_leaves && (static_cast<size_t>(c.skip - kids[k]) + 1) / 2 <= defer_leaves) {
                        w.child[k] = kWideEmpty;  // patched when the deferred subtrees are appended
                        deferred.push_back({kids[k], t.wnode, static_cast<uint32_t>(k), t.depth + 1});
                    } else {
                        const uint32_t wi = static_cast<uint32_t>(wide.size());
                        wide.emplace_back();
                        w.child[k] = wi;
                        todo.push_back({kids[k], wi, t.depth + 1});
                    }
                } else {
                    for (int a = 0; a < 3; ++a) {
                        w.plane[a][0][k] = std::numeric_limits<float>::infinity();
                        w.plane[a][1][k] = -std::numeric_limits<float>::infinity();
                        b64[k][a] = std::numeric_limits<double>::infinity(); b64[k][3 + a] = -std::numeric_limits<double>::infinity();
                    }
                    w.child[k] = kWideEmpty;
                }
            }
            wide[t.wnode] = w;
            if (boxes.size() < wide.size() * 24) boxes.resize(wide.size() * 24);
            std::memcpy(&boxes[static_cast<size_t>(t.wnode) * 24], b64, sizeof b64);
        }
        boxes.resize(wide.size() * 24);
    }
};

static void build_wide(const std::vector<DNode>& bn, std::vector<DWide>* out_wide, std::vector<double>* out_boxes, uint32_t* out_depth) {
    const size_t n_leaves = (bn.size() + 1) / 2;
    // big scenes: the top of the tree is collapsed here, subtrees of <= n/64 leaves on the host cores, then appended in order
    // (the result does not depend on the number of threads)
    WideBuilder top{bn, n_leaves >= 262144 ? std::max<size_t>(4096, n_leaves / 64) : 0};
    top.run(0, 1);
    std::vector<WideBuilder> subs;
    subs.reserve(top.deferred.size());
    for (size_t k = 0; k < top.deferred.size(); ++k) subs.push_back(WideBuilder{bn, 0});
    if (!subs.empty()) {
        std::atomic<size_t> next{0};
        std::vector<std::thread> pool;
        const size_t workers = std::max<size_t>(1, std::min<size_t>(std::thread::hardware_concurrency(), 32));
        for (size_t w = 0; w < workers; ++w)
            pool.emplace_back([&] {
                for (size_t k = next.fetch_add(1); k < subs.size(); k = next.fetch_add(1)) subs[k].run(top.deferred[k].bnode, top.deferred[k].depth);
            });
        for (std::thread& t : pool) t.join();
    }
    size_t total = top.wide.size();
    for (const WideBuilder& sb : subs) total += sb.wide.size();
    out_wide->swap(top.wide);
    out_boxes->swap(top.boxes);
    out_wide->reserve(total);
    out_boxes->reserve(total * 24);
    *out_depth = top.depth;
    for (size_t k = 0; k < subs.size(); ++k) {
        const uint32_t base = static_cast<uint32_t>(out_wide->size());
        (*out_wide)[top.deferred[k].parent].child[top.deferred[k].slot] = base;
        for (DWide w : subs[k].wide) {
            for (int c = 0; c < 4; ++c)
                if (!(w.child[c] & kWideLeaf)) w.child[c] += base;  // internal child: local index -> global (kWideEmpty has the leaf bit set)
            out_wide->push_back(w);
        }
        out_boxes->insert(out_boxes->end(), subs[k].boxes.begin(), subs[k].boxes.end());
        *out_depth = std::max(*out_depth, subs[k].depth);
        std::vector<DWide>().swap(subs[k].wide);
        std::vector<double>().swap(subs[k].boxes);
    }
}

// Scene-side preparation of the any-order walk (rtp_device.cu trace_any_kernel, DESIGN.md §4b). Distance culling is exact only
// with a bound on how far a primitive's computed t (hittable.rs:51-57, 85-95) can fall below the computed slab entry of its own
// box; that bound grows with the primitive's extent (a triangle's edges, a sphere's |o - c|^2 - r^2 cancellation), so the
// outsized primitives of a scene - the ground sphere of the bunny scenes, a floor made of two huge triangles - are taken out
// of the culled set: up to kMaxBig "big" primitives are tested when the ray starts, before its walk, and skipped when the walk
// meets their leaves. A tree too deep for the shared-memory stack, or irregular boxes, and the scene keeps the in-order walk.

// the leaf words of the big primitives carry kWideBig: the walk skips them
static void mark_big(std::vector<DWide>& wide, const std::vector<uint8_t>& is_big) {
    for (DWide& w : wide)
        for (uint32_t& c : w.child)
            if (c != kWideEmpty && (c & kWideLeaf) && is_big[c & kWideSlotMask]) c |= kWideBig;
}

static void prepare_any_order(const Switches& sw, FlatScene* out) {
    out->any_ok = false;
    out->n_big = 0;
    const size_t n = out->prims.size();
    if (!out->boxes_finite || n == 0 || out->root_kind != RTP_ROOT_BVH || out->wide_depth > 48) return;
    std::vector<uint8_t> kind(n, 0);
    for (const DNode& nd : out->nodes)
        if (nd.prim != kNoPrim) kind[nd.prim] = static_cast<uint8_t>(nd.kind);
    auto extent = [&](size_t s) {
        const DPrim& p = out->prims[s];
        return std::fmax(p.bmax[0] - p.bmin[0], std::fmax(p.bmax[1] - p.bmin[1], p.bmax[2] - p.bmin[2]));
    };
    // outsized primitives: more than 16 times the median extent; the eight largest of them are "big"
    std::vector<double> ext(n);
    for (size_t s = 0; s < n; ++s) ext[s] = extent(s);
    std::vector<uint8_t> is_big(n, 0);
    {
        std::vector<double> tmp = ext;
        std::nth_element(tmp.begin(), tmp.begin() + tmp.size() / 2, tmp.end());
        const double cap = 16.0 * tmp[tmp.size() / 2];
        std::vector<std::pair<double, uint32_t>> over;
        for (size_t s = 0; s < n; ++s)
            if (ext[s] > cap) over.push_back({ext[s], static_cast<uint32_t>(s)});
        std::sort(over.begin(), over.end(), [](const auto& a, const auto& b) { return a.first != b.first ? a.first > b.first : a.second < b.second; });
        for (size_t k = 0; k < over.size() && out->n_big < kMaxBig; ++k) {
            out->big[out->n_big++] = over[k].second | (static_cast<uint32_t>(kind[over[k].second]) << 31);
            is_big[over[k].second] = 1;
        }
    }
    // scene constants of the slack bound (rtp_device.cu any_slack): triangles E, A; spheres C (largest |centre coordinate|, bounded
    // by the box planes) and R (largest radius) - over the primitives that are not big; and the union of their boxes, which a ray
    // must enter within its window to need a walk at all (DSceneView::cull)
    double E = 0.0, A = 0.0, Cs = 0.0, Rs = 0.0;
    double ulo[3] = {std::numeric_limits<double>::infinity(), std::numeric_limits<double>::infinity(), std::numeric_limits<double>::infinity()};
    double uhi[3] = {-ulo[0], -ulo[1], -ulo[2]};
    bool spheres = false;
    for (size_t s = 0; s < n; ++s) {
        if (is_big[s]) continue;
        const DPrim& p = out->prims[s];
        double mag = 0.0;
        for (int k = 0; k < 3; ++k) mag = std::fmax(mag, std::fmax(std::fabs(p.bmin[k]), std::fabs(p.bmax[k])));
        for (int k = 0; k < 3; ++k) { ulo[k] = std::fmin(ulo[k], p.bmin[k]); uhi[k] = std::fmax(uhi[k], p.bmax[k]); }
        if (kind[s] == RTP_HITTABLE_SPHERE) {
            spheres = true;
            Cs = std::fmax(Cs, mag);
            Rs = std::fmax(Rs, 0.5 * ext[s]);
        } else {
            E = std::fmax(E, ext[s]);
            A = std::fmax(A, mag);
        }
    }
    out->any_E = E * (1.0 + 1e-12);
    out->any_A = A * (1.0 + 1e-12);
    out->any_spheres = spheres;
    out->any_C = Cs * (1.0 + 1e-12);
    out->any_R = Rs * (1.0 + 1e-12);
    culled_set_box(ulo, uhi, out->cull);
    mark_big(out->wide, is_big);
    out->any_ok = true;

    if (n >= 2 && n > out->n_big && want_free_tree(sw, n)) build_free_tree(out->prims[0].bmin, out->prims[0].bmax, sizeof(DPrim) / sizeof(double), kind, is_big, out);
}

// Free tree. The any-order walk does not need its leaves in the reference's depth-first order (only the re-walk does), so
// its lanes may walk a second culling tree built over the MORTON order of the leaf centroids with the same SAH-over-a-sequence
// builder and the same 4-wide collapse; its leaves carry the same slots. Measured: 4-6 % faster on the bunny (4.06 instead of
// 4.26 nodes per primary ray, 4 ms of build), no gain on the bunny fields (15.4 instead of 15.6 nodes, 1.5 s of build for
// 2.5 M leaves) - so only scenes below kFreeTreeLeaves get it by default. It holds only the primitives that are not big: those
// are tested before the walk starts, and left out the root box no longer spans the ground sphere that every ray enters.
void build_free_tree(const double* bmin, const double* bmax, size_t stride, const std::vector<uint8_t>& kind, const std::vector<uint8_t>& is_big,
                     FlatScene* out) {
    const size_t n = kind.size(), m = n - out->n_big;
    auto lo_of = [&](size_t s) { return bmin + s * stride; };
    auto hi_of = [&](size_t s) { return bmax + s * stride; };
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (size_t s = 0; s < n; ++s) {
        if (is_big[s]) continue;
        for (int k = 0; k < 3; ++k) { const double c = 0.5 * (lo_of(s)[k] + hi_of(s)[k]); lo[k] = std::fmin(lo[k], c); hi[k] = std::fmax(hi[k], c); }
    }
    auto spread = [](uint64_t x) {  // 21 bits -> every third bit
        x &= 0x1FFFFFull;
        x = (x | x << 32) & 0x1F00000000FFFFull; x = (x | x << 16) & 0x1F0000FF0000FFull; x = (x | x << 8) & 0x100F00F00F00F00Full;
        x = (x | x << 4) & 0x10C30C30C30C30C3ull; x = (x | x << 2) & 0x1249249249249249ull;
        return x;
    };
    std::vector<std::pair<uint64_t, uint32_t>> keyed(n);
    parallel_chunks(n, [&](size_t a, size_t b) {
        for (size_t s = a; s < b; ++s) {
            uint64_t key = 0;  // big primitives sort first and are dropped below
            if (!is_big[s]) {
                uint64_t q[3];
                for (int k = 0; k < 3; ++k) {
                    const double c = 0.5 * (lo_of(s)[k] + hi_of(s)[k]), ext = hi[k] - lo[k];
                    const double f = ext > 0.0 ? (c - lo[k]) / ext : 0.0;
                    q[k] = static_cast<uint64_t>(std::fmin(std::fmax(f, 0.0), 1.0) * 2097151.0);
                }
                key = (uint64_t(1) << 63) | spread(q[0]) | spread(q[1]) << 1 | spread(q[2]) << 2;
            }
            keyed[s] = {key, static_cast<uint32_t>(s)};
        }
    });
    std::sort(keyed.begin(), keyed.end());
    std::vector<BuildItem> seq(m);
    for (size_t i = 0; i < m; ++i) {
        const uint32_t s = keyed[out->n_big + i].second;
        seq[i].id = s;
        std::memcpy(seq[i].bmin, lo_of(s), sizeof seq[i].bmin);
        std::memcpy(seq[i].bmax, hi_of(s), sizeof seq[i].bmax);
    }
    std::vector<DNode> nodes(2 * m - 1);
    SeqBuilder sb{seq, nodes};
    sb.build(0, m, 0, 1, 4);
    for (DNode& nd : nodes)
        if (nd.prim != kNoPrim) { const uint32_t slot = seq[nd.prim].id; nd.prim = slot; nd.kind = kind[slot]; }
    build_wide(nodes, &out->free_wide, &out->free_boxes, &out->free_depth);
}

static bool emit_ok(const rtp_emit& e, uint32_t n_textures) {
    if (e.kind > RTP_EMIT_SKY_SPHERE) return false;
    return e.kind != RTP_EMIT_SKY_SPHERE || e.texture < n_textures;
}

// ---------------------------------------------------------------------------------------------
// Nested containers (hittable.rs:13-14: `List` and `Bvh` as items of another container). Everything the reference does with
// them is again a SEQUENTIAL process over primitives: hit_list (hittable.rs:110-120) tests its items in order against the
// shrinking ray and lets a later hit replace an earlier one; a Bvh leaf that holds a List is gated by the List's union box
// (hittable.rs:142-147) and then runs that list; a Bvh inside a List is its own Bvh::hit, i.e. its leaves in its own
// depth-first order, each behind its own box. So a scene with nesting flattens to one sequence of primitives, each with the
// box that gates it (or none): exactly the form `Bvh::hit ≡ for leaf in order: if collide(gate) and hit(prim)` that
// DESIGN.md §2 derives for the flat case. The reported leaf id is the index of the root container's item that holds the winner.
// ---------------------------------------------------------------------------------------------
struct SeqPrim {
    const rtp_hittable* h;
    uint32_t top;   // index of the root container's item this primitive belongs to
    bool gated;
    double gmin[3], gmax[3];
};

struct NestedFlattener {
    const rtp_scene_desc* d;
    std::vector<SeqPrim> seq;
    int err = RTP_OK;
    std::string msg;
    uint32_t root_depth = 0;

    void fail(int code, const std::string& m) { if (err == RTP_OK) { err = code; msg = m; } }

    bool check(const rtp_hittable* h, bool in_nested, uint32_t index) {
        if (h->kind == RTP_HITTABLE_SPHERE) { if (h->material >= d->n_materials) { fail(RTP_ERR_INVALID, "sphere material out of range"); return false; } }
        else if (h->kind == RTP_HITTABLE_TRIANGLE) {
            if (h->mesh >= d->n_meshes || static_cast<uint64_t>(h->triangle) + 3 > d->meshes[h->mesh].n_indices) { fail(RTP_ERR_INVALID, "triangle id out of range"); return false; }
        } else if (h->kind == RTP_HITTABLE_LIST || h->kind == RTP_HITTABLE_BVH) {
            // a run of `nested`; a nested container's run lies entirely before the container itself, so nesting cannot cycle
            if (static_cast<uint64_t>(h->mesh) + h->triangle > (in_nested ? index : d->n_nested)) { fail(RTP_ERR_INVALID, "nested run out of range"); return false; }
            if (h->kind == RTP_HITTABLE_BVH && h->triangle == 0) { fail(RTP_ERR_INVALID, "Bvh::new on an empty list is unreachable!() in the reference (bvh.rs:40)"); return false; }
        } else { fail(RTP_ERR_INVALID, "unknown hittable kind"); return false; }
        return true;
    }

    // hittable.rs:27-34, 124-147; false where the reference panics (the box of a Bvh, hittable.rs:32)
    bool bbox(const rtp_hittable* h, double* lo, double* hi) {
        if (h->kind == RTP_HITTABLE_BVH) { fail(RTP_ERR_INVALID, "bounding box of a Bvh: \"Do not take the bounding box of a Bvh\" (hittable.rs:32)"); return false; }
        if (h->kind == RTP_HITTABLE_LIST) {  // AABB::default() when empty, else a left fold of AABB::union (utility.rs:130-135)
            for (int k = 0; k < 3; ++k) lo[k] = hi[k] = 0.0;
            const rtp_hittable* items = d->nested + h->mesh;
            for (uint32_t i = 0; i < h->triangle; ++i) {
                double a[3], b[3];
                if (!bbox(&items[i], a, b)) return false;
                for (int k = 0; k < 3; ++k) { lo[k] = i ? min_num(lo[k], a[k]) : a[k]; hi[k] = i ? max_num(hi[k], b[k]) : b[k]; }
            }
            return true;
        }
        if (h->kind == RTP_HITTABLE_SPHERE) {
            for (int k = 0; k < 3; ++k) { lo[k] = h->center[k] - h->radius; hi[k] = h->center[k] + h->radius; }
            return true;
        }
        const rtp_mesh& m = d->meshes[h->mesh];
        const double* a = m.vertices[m.indices[h->triangle + 0]].position;
        const double* b = m.vertices[m.indices[h->triangle + 1]].position;
        const double* c = m.vertices[m.indices[h->triangle + 2]].position;
        for (int k = 0; k < 3; ++k) { lo[k] = min_num(min_num(a[k], b[k]), c[k]); hi[k] = max_num(max_num(a[k], b[k]), c[k]); }
        return true;
    }

    // the primitives of `h` in evaluation order, all behind `gate` (nullptr: none)
    void emit(const rtp_hittable* h, uint32_t top, const double* gate) {
        if (err != RTP_OK) return;
        if (h->kind == RTP_HITTABLE_LIST) {
            const rtp_hittable* items = d->nested + h->mesh;
            for (uint32_t i = 0; i < h->triangle; ++i) emit(&items[i], top, gate);
        } else if (h->kind == RTP_HITTABLE_BVH) {
            if (gate) { fail(RTP_ERR_INVALID, "a Bvh below a Bvh leaf: its bounding box is needed (hittable.rs:32 panics)"); return; }
            emit_bvh(d->nested + h->mesh, h->triangle, false, top);
        } else {
            SeqPrim sp;
            sp.h = h; sp.top = top; sp.gated = gate != nullptr;
            for (int k = 0; k < 3; ++k) { sp.gmin[k] = gate ? gate[k] : 0.0; sp.gmax[k] = gate ? gate[3 + k] : 0.0; }
            seq.push_back(sp);
        }
    }

    // Bvh::new (bvh.rs:70-91) over `items`, then its leaves in depth-first order, each behind its own box
    void emit_bvh(const rtp_hittable* items, uint32_t n, bool is_root, uint32_t top) {
        std::vector<BuildItem> bi(n);
        for (uint32_t i = 0; i < n && err == RTP_OK; ++i) {
            bi[i].id = i;
            if (!bbox(&items[i], bi[i].bmin, bi[i].bmax)) return;
            for (int k = 0; k < 3; ++k) {
                const double key = 0.5 * (bi[i].bmin[k] + bi[i].bmax[k]);
                if (key != key) { fail(RTP_ERR_INVALID, "NaN bounding-box centroid (partial_cmp().unwrap() panics, bvh.rs:63)"); return; }
            }
        }
        if (err != RTP_OK) return;
        std::vector<DNode> tmp(static_cast<size_t>(2) * n - 1);
        Builder b{bi, tmp};
        b.build(0, n, 0, 0, 1, 0);
        if (is_root) root_depth = b.depth.load();
        for (uint32_t r = 0; r < n; ++r) {
            double gate[6];
            for (int k = 0; k < 3; ++k) { gate[k] = bi[r].bmin[k]; gate[3 + k] = bi[r].bmax[k]; }
            emit(&items[bi[r].id], is_root ? bi[r].id : top, gate);
        }
    }
};

int flatten_scene(const rtp_scene_desc* d, const Switches& sw, FlatScene* out, bool device_build) {
    if (!d || !out) return set_error(RTP_ERR_INVALID, "null scene description");
    if (d->abi_version != RTP_ABI_VERSION) return set_error(RTP_ERR_INVALID, "rtp_scene_desc.abi_version mismatch");
    if (d->root_kind > RTP_ROOT_LIST) return set_error(RTP_ERR_INVALID, "unknown root kind");
    if ((d->n_meshes && !d->meshes) || (d->n_hittables && !d->hittables) || (d->n_materials && !d->materials) ||
        (d->n_textures && !d->textures))
        return set_error(RTP_ERR_INVALID, "null table with non-zero count");
    if (d->root_kind == RTP_ROOT_BVH && d->n_hittables == 0)
        return set_error(RTP_ERR_INVALID, "Bvh::new on an empty list is unreachable!() in the reference (bvh.rs:40)");
    if (d->n_hittables >= kWideSlotMask) return set_error(RTP_ERR_INVALID, "too many hittables");

    auto t0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!sw.build_timing) return;
        auto t1 = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[rtp build] %s: %.3f s\n", what, std::chrono::duration<double>(t1 - t0).count());
        t0 = t1;
    };

    // ---- tables -------------------------------------------------------------------------
    out->root_kind = d->root_kind;
    out->background = d->background;
    if (!emit_ok(d->background, d->n_textures)) return set_error(RTP_ERR_INVALID, "background emit is invalid");
    out->textures.resize(d->n_textures);
    out->images.resize(d->n_textures);
    for (uint32_t i = 0; i < d->n_textures; ++i) {
        const rtp_texture& t = d->textures[i];
        if (t.kind > RTP_TEXTURE_PERLIN) return set_error(RTP_ERR_INVALID, "unknown texture kind");
        DTexture& o = out->textures[i];
        std::memset(&o, 0, sizeof o);
        o.kind = t.kind; o.width = t.width; o.height = t.height; o.odd = t.odd; o.even = t.even; o.seed = t.seed;
        std::memcpy(o.rgb, t.rgb, sizeof o.rgb);
        if (t.kind == RTP_TEXTURE_IMAGE) {
            size_t bytes = static_cast<size_t>(t.width) * t.height * 4;
            if (!t.rgba || bytes == 0) return set_error(RTP_ERR_INVALID, "image texture without texels");
            out->images[i].assign(t.rgba, t.rgba + bytes);
        }
        if (t.kind == RTP_TEXTURE_CHECKER && (t.odd >= d->n_textures || t.even >= d->n_textures))
            return set_error(RTP_ERR_INVALID, "checker texture id out of range");
    }
    out->materials.resize(d->n_materials);
    for (uint32_t i = 0; i < d->n_materials; ++i) {
        const rtp_material& m = d->materials[i];
        if (m.scatter > RTP_SCATTER_DIELECTRIC || m.absorb > RTP_ABSORB_ALBEDO_MAP || !emit_ok(m.emit, d->n_textures) ||
            (m.absorb == RTP_ABSORB_ALBEDO_MAP && m.absorb_texture >= d->n_textures))
            return set_error(RTP_ERR_INVALID, "material " + std::to_string(i) + " is invalid");
        DMaterial& o = out->materials[i];
        std::memset(&o, 0, sizeof o);
        o.scatter = m.scatter; o.absorb = m.absorb; o.absorb_texture = m.absorb_texture;
        o.emit_kind = m.emit.kind; o.emit_texture = m.emit.texture;
        o.scatter_param = m.scatter_param;
        std::memcpy(o.absorb_rgb, m.absorb_rgb, sizeof o.absorb_rgb);
        std::memcpy(o.emit_rgb, m.emit.rgb, sizeof o.emit_rgb);
    }
    for (uint32_t i = 0; i < d->n_meshes; ++i) {
        const rtp_mesh& m = d->meshes[i];
        if ((m.n_vertices && !m.vertices) || (m.n_indices && !m.indices)) return set_error(RTP_ERR_INVALID, "null mesh arrays");
        if (m.material >= d->n_materials) return set_error(RTP_ERR_INVALID, "mesh material out of range");
        for (uint32_t k = 0; k < m.n_indices; ++k)
            if (m.indices[k] >= m.n_vertices) return set_error(RTP_ERR_INVALID, "vertex index out of range");
    }

    // ---- leaf boxes: hittable.rs:124-140 ---------------------------------------------------
    if (d->n_nested && !d->nested) return set_error(RTP_ERR_INVALID, "null nested table with non-zero count");
    bool nested = false;
    for (uint32_t i = 0; i < d->n_hittables && !nested; ++i) nested = d->hittables[i].kind >= RTP_HITTABLE_LIST;
    uint32_t n = d->n_hittables;      // primitives of the flattened scene (more than n_hittables when containers are nested)
    std::vector<BuildItem> items;     // per primitive slot: the box that gates it + the id reported for it
    std::vector<const rtp_hittable*> prim_h;  // per primitive slot: its Sphere / Triangle description
    std::vector<uint8_t> gated;       // nested List roots: the primitive sits behind a box (a leaf of a nested Bvh)
    NestedFlattener nf{d};
    // Big flat Bvh scenes are built on the device from here on (rtp_build.cu device_build_scene): leaf boxes, reference order, SAH
    // culling tree, records, 4-wide collapse and the any-order tables never exist on the host. RTP_DEVICE_BUILD: "0" never,
    // "1" always (tests compare both builds), unset: scenes of >= 65,536 leaves.
    if (device_build && !nested && d->root_kind == RTP_ROOT_BVH && n >= 2 && !sw.reference_tree) {
        if (sw.device_build >= 0 ? sw.device_build != 0 : n >= 65536u) {
            lap("tables and validation");
            const int rc = device_build_scene(d, sw, out);
            if (rc == RTP_OK) { lap("device build"); return RTP_OK; }
            if (rc != 1) return rc;
            // 1: not applicable (inverted or non-finite boxes): the host path below keeps the reference topology for such scenes
        }
    }
    if (nested) {
        for (uint32_t i = 0; i < d->n_hittables; ++i) if (!nf.check(&d->hittables[i], false, i)) return set_error(nf.err, nf.msg);
        for (uint32_t i = 0; i < d->n_nested; ++i) if (!nf.check(&d->nested[i], true, i)) return set_error(nf.err, nf.msg);
        if (d->root_kind == RTP_ROOT_BVH) nf.emit_bvh(d->hittables, d->n_hittables, true, 0);
        else for (uint32_t i = 0; i < d->n_hittables; ++i) nf.emit(&d->hittables[i], i, nullptr);
        if (nf.err != RTP_OK) return set_error(nf.err, nf.msg);
        if (nf.seq.size() >= kWideSlotMask) return set_error(RTP_ERR_INVALID, "too many primitives");
        n = static_cast<uint32_t>(nf.seq.size());
        if (d->root_kind == RTP_ROOT_BVH && n == 0) return set_error(RTP_ERR_UNSUPPORTED, "a Bvh whose leaves are all empty lists holds no primitive");
        items.resize(n); prim_h.resize(n); gated.resize(n);
        for (uint32_t k = 0; k < n; ++k) {
            const SeqPrim& sp = nf.seq[k];
            items[k].id = sp.top;
            std::memcpy(items[k].bmin, sp.gmin, sizeof sp.gmin);
            std::memcpy(items[k].bmax, sp.gmax, sizeof sp.gmax);
            prim_h[k] = sp.h;
            gated[k] = sp.gated ? 1 : 0;
        }
    } else {
    items.resize(n);
    // the error of the smallest failing index, whichever chunk finds it first (the device build reports the same one): a chunk
    // stops at its first failure, or once a smaller failing index is known
    std::atomic<uint32_t> first_bad{std::numeric_limits<uint32_t>::max()};
    int bad_code = RTP_OK;
    std::string bad_msg;
    std::mutex bad_lock;
    auto fail = [&](uint32_t i, int code, const std::string& msg) {
        std::lock_guard<std::mutex> g(bad_lock);
        if (i < first_bad.load()) { first_bad.store(i); bad_code = code; bad_msg = msg; }
    };
    parallel_chunks(n, [&](size_t lo_i, size_t hi_i) {
      for (uint32_t i = static_cast<uint32_t>(lo_i); i < hi_i && i < first_bad.load(std::memory_order_relaxed); ++i) {
        const rtp_hittable& h = d->hittables[i];
        BuildItem& it = items[i];
        it.id = i;
        if (h.kind == RTP_HITTABLE_SPHERE) {
            if (h.material >= d->n_materials) { fail(i, RTP_ERR_INVALID, "sphere material out of range"); return; }
            for (int k = 0; k < 3; ++k) {
                it.bmin[k] = h.center[k] - h.radius;
                it.bmax[k] = h.center[k] + h.radius;
            }
        } else if (h.kind == RTP_HITTABLE_TRIANGLE) {
            if (h.mesh >= d->n_meshes || static_cast<uint64_t>(h.triangle) + 3 > d->meshes[h.mesh].n_indices)
                { fail(i, RTP_ERR_INVALID, "triangle id out of range"); return; }
            const rtp_mesh& m = d->meshes[h.mesh];
            const double* a = m.vertices[m.indices[h.triangle + 0]].position;
            const double* b = m.vertices[m.indices[h.triangle + 1]].position;
            const double* c = m.vertices[m.indices[h.triangle + 2]].position;
            for (int k = 0; k < 3; ++k) {
                it.bmin[k] = min_num(min_num(a[k], b[k]), c[k]);
                it.bmax[k] = max_num(max_num(a[k], b[k]), c[k]);
            }
        } else {
            { fail(i, RTP_ERR_INVALID, "unknown hittable kind"); return; }
        }
        if (d->root_kind == RTP_ROOT_BVH)
            for (int k = 0; k < 3; ++k) {
                double key = 0.5 * (it.bmin[k] + it.bmax[k]);
                if (key != key)  // partial_cmp().unwrap() panics on NaN (bvh.rs:63)
                    { fail(i, RTP_ERR_INVALID, "NaN bounding-box centroid in hittable " + std::to_string(i)); return; }
            }
      }
    });
    if (bad_code != RTP_OK) return set_error(bad_code, bad_msg);
    }

    // ---- tree ---------------------------------------------------------------------------------
    out->depth = 0;
    if (d->root_kind == RTP_ROOT_BVH && nested) {
        // the sequence is already in evaluation order (NestedFlattener); any binary tree over it is a valid culling tree as long
        // as every gate box is ordered and finite (DESIGN.md §2), so the SAH-over-a-sequence builder is used directly
        for (const BuildItem& it : items)
            for (int k = 0; k < 3; ++k)
                if (!(it.bmin[k] <= it.bmax[k]) || !std::isfinite(it.bmin[k]) || !std::isfinite(it.bmax[k]))
                    return set_error(RTP_ERR_UNSUPPORTED, "nested containers together with an inverted or non-finite bounding box");
        out->nodes.assign(static_cast<size_t>(2) * n - 1, DNode{});
        out->depth = nf.root_depth;
        out->n_reference_nodes = 2 * d->n_hittables - 1;
        SeqBuilder sb{items, out->nodes};
        sb.build(0, n, 0, 1, 4);
        out->device_depth = sb.depth.load();
        lap("nested containers flattened; SAH culling tree over the evaluation order");
    } else if (d->root_kind == RTP_ROOT_BVH) {
        out->nodes.assign(static_cast<size_t>(2) * n - 1, DNode{});
        lap("tables, validation, leaf boxes");
        Builder b{items, out->nodes};
        b.build(0, n, 0, 0, 1, 4);  // sorts `items` into the reference's DFS-rank order
        lap("reference median-split order (Bvh::new)");
        out->depth = b.depth.load();
        out->n_reference_nodes = static_cast<uint32_t>(out->nodes.size());
        // The freedom to re-shape the tree (DESIGN.md §2) rests on ordered, finite leaf boxes (min <= max on every axis: a
        // parent's slab interval then contains each child's). A sphere of negative radius has an INVERTED box (hittable.rs:124-131
        // computes center -/+ radius), which AABB::collide still treats like the proper box but AABB::union does not, so what the
        // reference returns for such a scene depends on its own topology: keep that topology and the literal slab test.
        bool regular = true;
        for (const BuildItem& it : items)
            for (int k = 0; k < 3; ++k)
                if (!(it.bmin[k] <= it.bmax[k]) || !std::isfinite(it.bmin[k]) || !std::isfinite(it.bmax[k])) regular = false;
        if (!regular) out->boxes_finite = false;
        if (regular && !sw.reference_tree) {  // RTP_TREE=reference keeps the median-split topology on the device (A/B runs, counter parity)
            SeqBuilder sb{items, out->nodes};
            sb.build(0, n, 0, 1, 4);
            out->device_depth = sb.depth.load();
            lap("SAH culling tree over the rank order");
        } else {
            out->device_depth = out->depth;
        }
    }
    for (const DNode& nd : out->nodes)
        for (int k = 0; k < 3; ++k) {
            if (!std::isfinite(nd.bmin[k]) || !std::isfinite(nd.bmax[k])) out->boxes_finite = false;
            out->scene_mag = std::fmax(out->scene_mag, std::fmax(std::fabs(nd.bmin[k]), std::fabs(nd.bmax[k])));
        }
    // List roots keep the caller's order (hittable.rs:113); Bvh roots are now in DFS-rank order.

    // ---- primitives in traversal order ----------------------------------------------------------
    out->prims.resize(n);
    out->attrs.resize(n);
    out->leaf_order.resize(n);
    parallel_chunks(n, [&](size_t lo_s, size_t hi_s) {
      for (uint32_t slot = static_cast<uint32_t>(lo_s); slot < hi_s; ++slot) {
        uint32_t id = items[slot].id;
        const rtp_hittable& h = nested ? *prim_h[slot] : d->hittables[id];
        DPrim& p = out->prims[slot];
        DAttr& at = out->attrs[slot];
        std::memset(&p, 0, sizeof p);
        std::memset(&at, 0, sizeof at);
        p.leaf = id;
        out->leaf_order[slot] = id;
        std::memcpy(p.bmin, items[slot].bmin, sizeof p.bmin);  // hittable.rs:124-140, the leaf's own gate box
        std::memcpy(p.bmax, items[slot].bmax, sizeof p.bmax);
        if (h.kind == RTP_HITTABLE_SPHERE) {
            for (int k = 0; k < 3; ++k) p.a[k] = h.center[k];
            p.ba[0] = h.radius;
            p.material = h.material;
        } else {
            const rtp_mesh& m = d->meshes[h.mesh];
            const rtp_vertex& va = m.vertices[m.indices[h.triangle + 0]];
            const rtp_vertex& vb = m.vertices[m.indices[h.triangle + 1]];
            const rtp_vertex& vc = m.vertices[m.indices[h.triangle + 2]];
            for (int k = 0; k < 3; ++k) {
                p.a[k] = va.position[k];
                p.ba[k] = va.position[k] - vb.position[k];  // hittable.rs:71
                p.ca[k] = va.position[k] - vc.position[k];  // hittable.rs:72
                at.n[0][k] = va.normal[k];
                at.n[1][k] = vb.normal[k];
                at.n[2][k] = vc.normal[k];
            }
            for (int k = 0; k < 2; ++k) {
                at.uv[0][k] = va.uv[k];
                at.uv[1][k] = vb.uv[k];
                at.uv[2][k] = vc.uv[k];
            }
            p.material = m.material;  // hittable.rs:107
        }
      }
    });
    lap("primitive and attribute records");
    if (d->root_kind == RTP_ROOT_BVH) {
        for (DNode& nd : out->nodes)
            if (nd.prim != kNoPrim) nd.kind = nested ? prim_h[nd.prim]->kind : d->hittables[items[nd.prim].id].kind;
        build_wide(out->nodes, &out->wide, &out->wide_boxes, &out->wide_depth);
        lap("4-wide collapse");
        prepare_any_order(sw, out);
        lap(out->free_wide.empty() ? "any-order walk tables" : "any-order walk tables and the order-free culling tree");
    } else {
        // a List root is traversed as a flat run of leaves without slab tests; nodes carry only the kind
        out->nodes.assign(n ? n : 1, DNode{});
        for (uint32_t slot = 0; slot < n; ++slot) {
            DNode& nd = out->nodes[slot];
            nd.skip = slot + 1; nd.prim = slot; nd.kind = nested ? prim_h[slot]->kind : d->hittables[slot].kind;
            nd._pad = (nested && gated[slot]) ? 1u : 0u;  // the primitive sits behind the box in its DPrim (leaf of a nested Bvh): gate it first
            if (nd._pad) out->list_gates = true;
        }
        if (n == 0) { out->nodes[0].skip = 1; out->nodes[0].prim = kNoPrim; }
    }
    return RTP_OK;
}

// --------------------------------------------------------------------------- OBJ -----------------

namespace {

struct ObjCorner {
    uint32_t p, n, t;  // n, t == RTP_MISS when absent
    bool operator==(const ObjCorner& o) const { return p == o.p && n == o.n && t == o.t; }
};
struct ObjCornerHash {
    size_t operator()(const ObjCorner& c) const {
        uint64_t h = c.p * 0x9E3779B97F4A7C15ull;
        h ^= (h >> 29) + c.n * 0xBF58476D1CE4E5B9ull;
        h ^= (h >> 31) + c.t * 0x94D049BB133111EBull;
        return static_cast<size_t>(h ^ (h >> 32));
    }
};

struct Cursor {
    const char* p;
    const char* end;
    bool zero_index = false;  // a face corner named index 0: OBJ indices are 1-based, the reference's `- 1` (mesh.rs:64-69) underflows and panics
    bool blank() const { return p < end && (*p == ' ' || *p == '\t'); }
    // nom `space1`
    bool space1() {
        if (!blank()) return false;
        while (blank()) ++p;
        return true;
    }
    // nom `double`: no leading whitespace allowed
    bool real(double* out) {
        if (p >= end || blank() || *p == '\r' || *p == '\n') return false;
        char* e = nullptr;
        double v = std::strtod(p, &e);
        if (e == p) return false;
        p = e;
        *out = v;
        return true;
    }
    bool reals(double* out, int n) {
        for (int k = 0; k < n; ++k) {
            if (k && !space1()) return false;
            if (!real(&out[k])) return false;
        }
        return true;
    }
    // mesh.rs:58-70: separated_list1("/", opt(integer)); [0] position (required), [1] texcoord, [2] normal
    bool corner(ObjCorner* out) {
        uint32_t val[3] = {0, 0, 0};
        bool have[3] = {false, false, false};
        const char* q = p;
        for (int field = 0;; ++field) {
            uint64_t v = 0;
            int digits = 0;
            while (q < end && *q >= '0' && *q <= '9') {
                v = v * 10 + static_cast<uint64_t>(*q - '0');
                if (v > 0xFFFFFFFFull) return false;
                ++q; ++digits;
            }
            if (field < 3) { have[field] = digits > 0; val[field] = static_cast<uint32_t>(v); }
            if (q < end && *q == '/') { ++q; continue; }
            break;
        }
        if (!have[0]) return false;
        for (int k = 0; k < 3; ++k)
            if (have[k] && val[k] == 0) zero_index = true;
        out->p = val[0] - 1;
        out->t = have[1] ? val[1] - 1 : RTP_MISS;
        out->n = have[2] ? val[2] - 1 : RTP_MISS;
        p = q;
        return true;
    }
};

}  // namespace

static int obj_load(const char* path, rtp_mesh* out) {
    std::ifstream f(path, std::ios::binary);
    if (!f) return set_error(RTP_ERR_IO, std::string("cannot open ") + path);
    std::string text((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());

    std::vector<double> positions, normals, texcoords;  // flat xyz / xyz / uv
    std::vector<ObjCorner> corners;
    std::vector<std::pair<uint32_t, uint32_t>> faces;  // first corner, corner count

    const char* s = text.data();
    const char* end = s + text.size();
    while (s < end) {
        const char* eol = static_cast<const char*>(std::memchr(s, '\n', static_cast<size_t>(end - s)));
        if (!eol) eol = end;
        Cursor c{s, eol};
        double v[3];
        // mesh.rs:94-101: alt((v, vn, vt, f)); each is tag + space1 + payload, unparseable lines are skipped
        if (eol - s >= 2 && s[0] == 'v' && (s[1] == ' ' || s[1] == '\t')) {
            c.p = s + 1;
            if (c.space1() && c.reals(v, 3)) positions.insert(positions.end(), v, v + 3);
        } else if (eol - s >= 3 && s[0] == 'v' && s[1] == 'n') {
            c.p = s + 2;
            if (c.space1() && c.reals(v, 3)) normals.insert(normals.end(), v, v + 3);
        } else if (eol - s >= 3 && s[0] == 'v' && s[1] == 't') {
            c.p = s + 2;
            if (c.space1() && c.reals(v, 2)) texcoords.insert(texcoords.end(), v, v + 2);
        } else if (eol - s >= 2 && s[0] == 'f') {
            c.p = s + 1;
            if (c.space1()) {
                uint32_t first = static_cast<uint32_t>(corners.size()), count = 0;
                ObjCorner oc;
                while (c.corner(&oc)) {
                    corners.push_back(oc);
                    ++count;
                    if (!c.space1()) break;
                }
                if (c.zero_index) return set_error(RTP_ERR_FORMAT, "OBJ face with index 0: indices are 1-based (mesh.rs:64-69 would underflow)");
                if (count) faces.emplace_back(first, count);
            }
        }
        s = eol + 1;
    }

    // mesh.rs:151-166: one vertex per distinct (p, n, t), numbered in first-seen order
    std::unordered_map<ObjCorner, uint32_t, ObjCornerHash> unique;
    unique.reserve(corners.size());
    std::vector<rtp_vertex> vertices;
    std::vector<uint32_t> corner_vertex(corners.size());
    const size_t np = positions.size() / 3, nn = normals.size() / 3, nt = texcoords.size() / 2;
    for (size_t k = 0; k < corners.size(); ++k) {
        const ObjCorner& oc = corners[k];
        auto it = unique.find(oc);
        if (it != unique.end()) { corner_vertex[k] = it->second; continue; }
        if (oc.p >= np || (oc.n != RTP_MISS && oc.n >= nn) || (oc.t != RTP_MISS && oc.t >= nt))
            return set_error(RTP_ERR_FORMAT, "obj index out of range (the reference panics here)");
        rtp_vertex vx;
        std::memset(&vx, 0, sizeof vx);  // DEFAULT_NORMAL / DEFAULT_UV are zero (mesh.rs:146-147)
        std::memcpy(vx.position, &positions[3 * oc.p], 24);
        if (oc.n != RTP_MISS) std::memcpy(vx.normal, &normals[3 * oc.n], 24);
        if (oc.t != RTP_MISS) std::memcpy(vx.uv, &texcoords[2 * oc.t], 16);
        uint32_t id = static_cast<uint32_t>(vertices.size());
        unique.emplace(oc, id);
        vertices.push_back(vx);
        corner_vertex[k] = id;
    }
    std::vector<uint32_t> indices;
    indices.reserve(faces.size() * 3);
    for (const auto& fc : faces) {  // mesh.rs:169-179
        if (fc.second != 3) return set_error(RTP_ERR_FORMAT, "Non-triangular face are not supported");
        for (uint32_t k = 0; k < 3; ++k) indices.push_back(corner_vertex[fc.first + k]);
    }

    auto* vout = static_cast<rtp_vertex*>(std::malloc(sizeof(rtp_vertex) * std::max<size_t>(vertices.size(), 1)));
    auto* iout = static_cast<uint32_t*>(std::malloc(sizeof(uint32_t) * std::max<size_t>(indices.size(), 1)));
    if (!vout || !iout) { std::free(vout); std::free(iout); return set_error(RTP_ERR_NOMEM, "out of memory"); }
    if (!vertices.empty()) std::memcpy(vout, vertices.data(), sizeof(rtp_vertex) * vertices.size());
    if (!indices.empty()) std::memcpy(iout, indices.data(), sizeof(uint32_t) * indices.size());
    out->vertices = vout;
    out->indices = iout;
    out->n_vertices = static_cast<uint32_t>(vertices.size());
    out->n_indices = static_cast<uint32_t>(indices.size());
    out->material = 0;  // mesh.rs:181
    out->_pad = 0;
    return RTP_OK;
}

// --------------------------------------------------------------------------- TGA -----------------

static int tga_load(const char* path, rtp_image* out) {
    std::ifstream f(path, std::ios::binary);
    if (!f) return set_error(RTP_ERR_IO, std::string("cannot open ") + path);
    unsigned char hd[18];
    if (!f.read(reinterpret_cast<char*>(hd), 18)) return set_error(RTP_ERR_IO, "truncated tga header");
    const uint32_t w = hd[12] | (hd[13] << 8), h = hd[14] | (hd[15] << 8);
    const unsigned bpp = hd[16];
    const bool flip = (hd[17] & (1u << 5)) != 0;  // image.rs:95-99
    if (hd[0] != 0 || hd[1] != 0 || hd[2] != 2 || (bpp != 24 && bpp != 32))  // image.rs:81-88
        return set_error(RTP_ERR_FORMAT, "This tga header is not supported");
    const size_t src_px = bpp / 8, n = static_cast<size_t>(w) * h;
    std::vector<unsigned char> raw(n * src_px);
    if (n && !f.read(reinterpret_cast<char*>(raw.data()), static_cast<std::streamsize>(raw.size())))
        return set_error(RTP_ERR_IO, "truncated tga data");
    auto* rgba = static_cast<uint8_t*>(std::malloc(std::max<size_t>(n * 4, 1)));
    if (!rgba) return set_error(RTP_ERR_NOMEM, "out of memory");
    for (uint32_t row = 0; row < h; ++row) {
        const uint32_t dst_row = flip ? h - 1 - row : row;
        const unsigned char* src = raw.data() + static_cast<size_t>(row) * w * src_px;
        uint8_t* dst = rgba + static_cast<size_t>(dst_row) * w * 4;
        for (uint32_t x = 0; x < w; ++x, src += src_px, dst += 4) {
            dst[0] = src[2]; dst[1] = src[1]; dst[2] = src[0];
            dst[3] = src_px == 4 ? src[3] : 0xff;
        }
    }
    out->rgba = rgba; out->width = w; out->height = h;
    return RTP_OK;
}

static int tga_save(const rtp_image* img, const char* path) {
    if (img->width > 0xFFFFu || img->height > 0xFFFFu)
        return set_error(RTP_ERR_INVALID, "image dimensions do not fit a tga header (try_into fails, image.rs:123-124)");
    std::ofstream f(path, std::ios::binary);
    if (!f) return set_error(RTP_ERR_IO, std::string("cannot create ") + path);
    unsigned char hd[18] = {0};
    hd[2] = 2; hd[16] = 32;  // uncompressed BGRA, descriptor 0 = bottom-origin (image.rs:120-121)
    hd[12] = img->width & 0xff; hd[13] = img->width >> 8;
    hd[14] = img->height & 0xff; hd[15] = img->height >> 8;
    f.write(reinterpret_cast<const char*>(hd), 18);
    const size_t n = static_cast<size_t>(img->width) * img->height;
    std::vector<unsigned char> bgra(n * 4);
    for (size_t k = 0; k < n; ++k) {
        bgra[4 * k + 0] = img->rgba[4 * k + 2];
        bgra[4 * k + 1] = img->rgba[4 * k + 1];
        bgra[4 * k + 2] = img->rgba[4 * k + 0];
        bgra[4 * k + 3] = img->rgba[4 * k + 3];
    }
    f.write(reinterpret_cast<const char*>(bgra.data()), static_cast<std::streamsize>(bgra.size()));
    if (!f) return set_error(RTP_ERR_IO, "short write");
    return RTP_OK;
}

// --------------------------------------------------------------------------- Philox --------------

static void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
    for (int round = 0; round < 10; ++round) {
        const uint64_t m0 = 0xD2511F53ull * c[0], m1 = 0xCD9E8D57ull * c[2];
        const uint32_t x0 = static_cast<uint32_t>(m1 >> 32) ^ c[1] ^ k0;
        const uint32_t x2 = static_cast<uint32_t>(m0 >> 32) ^ c[3] ^ k1;
        c[0] = x0; c[1] = static_cast<uint32_t>(m1); c[2] = x2; c[3] = static_cast<uint32_t>(m0);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

}  // namespace rtp

// =============================================================================================
// C ABI — host-only entry points
// =============================================================================================

using namespace rtp;

extern "C" {

const char* rtp_last_error(void) { return g_last_error.c_str(); }
uint32_t rtp_abi_version(void) { return RTP_ABI_VERSION; }

int rtp_obj_load(const char* path, rtp_mesh* out) {
    if (!path || !out) return set_error(RTP_ERR_INVALID, "null argument");
    try { return obj_load(path, out); } catch (const std::exception& e) { return set_error(RTP_ERR_NOMEM, e.what()); }
}

void rtp_mesh_free(rtp_mesh* mesh) {
    if (!mesh) return;
    std::free(const_cast<rtp_vertex*>(mesh->vertices));
    std::free(const_cast<uint32_t*>(mesh->indices));
    mesh->vertices = nullptr; mesh->indices = nullptr;
    mesh->n_vertices = mesh->n_indices = 0;
}

int rtp_tga_load(const char* path, rtp_image* out) {
    if (!path || !out) return set_error(RTP_ERR_INVALID, "null argument");
    try { return tga_load(path, out); } catch (const std::exception& e) { return set_error(RTP_ERR_NOMEM, e.what()); }
}

int rtp_tga_save(const rtp_image* image, const char* path) {
    if (!image || !path || !image->rgba) return set_error(RTP_ERR_INVALID, "null argument");
    try { return tga_save(image, path); } catch (const std::exception& e) { return set_error(RTP_ERR_NOMEM, e.what()); }
}

void rtp_image_free(rtp_image* image) {
    if (!image) return;
    std::free(image->rgba);
    image->rgba = nullptr; image->width = image->height = 0;
}

int rtp_camera_lookat(const double position[3], const double target[3], const double up[3], rtp_camera* cam) {
    if (!position || !target || !up || !cam) return set_error(RTP_ERR_INVALID, "null argument");
    // utility.rs:172-177
    double d[3] = {position[0] - target[0], position[1] - target[1], position[2] - target[2]};
    const double len = std::sqrt(0.0 + dot3(d, d));
    const double z[3] = {d[0] / len, d[1] / len, d[2] / len};
    const double x[3] = {up[1] * z[2] - up[2] * z[1], up[2] * z[0] - up[0] * z[2], up[0] * z[1] - up[1] * z[0]};
    const double y[3] = {z[1] * x[2] - z[2] * x[1], z[2] * x[0] - z[0] * x[2], z[0] * x[1] - z[1] * x[0]};
    for (int r = 0; r < 3; ++r) {
        cam->orientation[0 + r] = x[r];
        cam->orientation[3 + r] = y[r];
        cam->orientation[6 + r] = z[r];
        cam->position[r] = position[r];
    }
    return RTP_OK;
}

int rtp_frame_to_srgb8(const double* rgb, uint32_t width, uint32_t height, uint8_t* out) {
    if (!rgb || !out) return set_error(RTP_ERR_INVALID, "null argument");
    const size_t n = static_cast<size_t>(width) * height;
    for (size_t p = 0; p < n; ++p) {
        for (int k = 0; k < 3; ++k) {  // utility.rs:212-220
            double x = rgb[3 * p + k];
            x = x < 0.0 ? 0.0 : (x > 1.0 ? 1.0 : x);  // f64::clamp keeps NaN
            const double y = 255.0 * std::pow(x, 1.0 / 2.2);
            out[4 * p + k] = !(y == y) || y <= 0.0 ? 0 : (y >= 255.0 ? 255 : static_cast<uint8_t>(y));  // `as u8` saturates
        }
        out[4 * p + 3] = 0xff;
    }
    return RTP_OK;
}

int rtp_split_in_tiles(uint32_t fw, uint32_t fh, uint32_t tw, uint32_t th, uint32_t* tiles, size_t cap, size_t* n) {
    if (!n || tw == 0 || th == 0) return set_error(RTP_ERR_INVALID, "bad tile arguments");
    // image.rs:151-167
    const uint32_t nti = (fw + tw - 1) / tw, ntj = (fh + th - 1) / th;
    size_t count = 0;
    for (uint32_t tj = 0; tj < ntj; ++tj)
        for (uint32_t ti = 0; ti < nti; ++ti, ++count) {
            if (!tiles || count >= cap) continue;
            const uint32_t oi = ti * tw, oj = tj * th;
            tiles[4 * count + 0] = oi;
            tiles[4 * count + 1] = oj;
            tiles[4 * count + 2] = std::min(tw, fw - oi);
            tiles[4 * count + 3] = std::min(th, fh - oj);
        }
    *n = count;
    return RTP_OK;
}

int rtp_rng_draws(uint64_t seed, uint32_t index_lo, uint32_t index_hi, uint32_t stream, uint32_t first_draw,
                  uint32_t n_draws, double* out) {
    if (n_draws && !out) return set_error(RTP_ERR_INVALID, "null argument");
    uint32_t cached = 0xFFFFFFFFu, block[4] = {0, 0, 0, 0};
    for (uint32_t i = 0; i < n_draws; ++i) {
        const uint32_t k = first_draw + i, b = k >> 1, pair = k & 1u;
        if (b != cached) {
            block[0] = index_lo; block[1] = index_hi; block[2] = b; block[3] = stream;
            philox4x32_10(block, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
            cached = b;
        }
        const uint64_t u = (static_cast<uint64_t>(block[2 * pair + 1]) << 32) | block[2 * pair];
        out[i] = static_cast<double>(u >> 11) * 0x1.0p-53;
    }
    return RTP_OK;
}

}  // extern "C"

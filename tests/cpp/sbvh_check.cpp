// CPU check and cost counter for the host SAH builder's spatial splits (csrc/bvh_sah.cpp; tests/test_sbvh_host.py).
//
//   sbvh_check TRIS RAYS [n_rays]
//     TRIS: n x 9 f64 (v0, v1, v2 of each triangle), RAYS: m x 7 f64 (o, d, t_max), raw little-endian
//     environment: T = builder threads (0 = all), RRT_SBVH_ALPHA / RRT_SBVH_CAP = the spatial-split parameters
//
// It builds the object-split tree (build_sah over the boxes alone) and the spatial-split tree (build_sah given the
// vertices), checks the spatial one — child boxes nested, subtree totals right, every triangle referenced, points sampled
// on every triangle inside a leaf that references it — and walks the rays through both in f64 the way the trace kernel
// does: both child boxes of an interior node are tested against [0, closest t so far], the nearer hit child is taken
// first, the other pushed; a leaf tests all its references with the kernel's Möller–Trumbore and accept rule.  It prints
// the mean interior visits and leaf tests per ray for both trees, and whether the closest hits (prim id, t bits) agree.
// (The kernel parks leaves and tests them a few steps late, and culls with fp32 boxes padded outward: its counts are
// somewhat higher than these.  The comparison between trees is what the counter is for.)
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>
#include "bvh_sah.hpp"
using namespace rrt;

static std::vector<double> read_f64(const char* path) {
    FILE* f = fopen(path, "rb");
    if (!f) {
        fprintf(stderr, "cannot open %s\n", path);
        exit(3);
    }
    fseek(f, 0, SEEK_END);
    const long bytes = ftell(f);
    fseek(f, 0, SEEK_SET);
    std::vector<double> v((size_t)bytes / sizeof(double));
    if (fread(v.data(), sizeof(double), v.size(), f) != v.size()) exit(3);
    fclose(f);
    return v;
}

// triangle.rs:233-265 as the trace kernel evaluates it (aggregate.cu tri_test; built with -ffp-contract=off)
static bool tri_test(const double* o, const double* d, const double* v, double* t) {
    double e1[3], e2[3], T[3], P[3], Q[3];
    for (int k = 0; k < 3; ++k) {
        e1[k] = v[3 + k] - v[k];
        e2[k] = v[6 + k] - v[k];
        T[k] = o[k] - v[k];
    }
    auto cross = [](const double* a, const double* b, double* c) {
        c[0] = a[1] * b[2] - a[2] * b[1];
        c[1] = a[2] * b[0] - a[0] * b[2];
        c[2] = a[0] * b[1] - a[1] * b[0];
    };
    auto dot = [](const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; };
    cross(d, e2, P);
    const double a = dot(e1, P);
    if (a > -0.0000001 && a < 0.0000001) return false;
    const double f = 1.0 / a;
    const double u = f * dot(T, P);
    if (u < 0.0 || u > 1.0) return false;
    cross(T, e1, Q);
    const double vv = f * dot(d, Q);
    if (vv < 0.0 || u + vv > 1.0) return false;
    const double tt = f * dot(e2, Q);
    if (tt < 0.0000001) return false;
    *t = tt;
    return true;
}

static bool slab(const double* o, const double* inv, const Aabb& b, double t_far, double* t_near) {
    double t0 = 0.0, t1 = t_far;
    for (int k = 0; k < 3; ++k) {
        double a = (b.lo[k] - o[k]) * inv[k], c = (b.hi[k] - o[k]) * inv[k];
        if (a > c) std::swap(a, c);
        if (!(a <= t1) || !(c >= t0)) return false;  // (the rays here have no zero direction component)
        t0 = std::max(t0, a);
        t1 = std::min(t1, c);
    }
    *t_near = t0;
    return t0 <= t1;
}

struct Walk {
    uint32_t prim = 0xFFFFFFFFu;
    double t = INFINITY;
    uint32_t visits = 0, tests = 0;
};

static Walk closest(const Bvh2& tree, const double* tris, const double* ray) {
    const double* o = ray;
    const double* d = ray + 3;
    double inv[3];
    for (int k = 0; k < 3; ++k) inv[k] = 1.0 / d[k];
    Walk w;
    w.t = ray[6];
    uint32_t stack[128];
    int sp = 0;
    uint32_t node = tree.root;
    for (;;) {
        const Bvh2Node& nd = tree.nodes[node];
        if (nd.count == 0) {
            ++w.visits;
            double tl, tr;
            const bool hl = slab(o, inv, tree.nodes[nd.left].box, w.t, &tl), hr = slab(o, inv, tree.nodes[nd.right].box, w.t, &tr);
            if (hl && hr) {
                const bool swap = tr < tl;
                stack[sp++] = swap ? (uint32_t)nd.left : (uint32_t)nd.right;
                node = swap ? (uint32_t)nd.right : (uint32_t)nd.left;
                continue;
            }
            if (hl || hr) {
                node = hl ? (uint32_t)nd.left : (uint32_t)nd.right;
                continue;
            }
        } else {
            for (uint32_t k = 0; k < nd.count; ++k) {
                const uint32_t pid = tree.order[nd.first + k];
                ++w.tests;
                double t;
                if (tri_test(o, d, tris + 9 * (size_t)pid, &t) && !(t > w.t)) {
                    if (t < w.t || w.prim == 0xFFFFFFFFu || pid < w.prim) {
                        w.t = t;
                        w.prim = pid;
                    }
                }
            }
        }
        if (sp == 0) break;
        node = stack[--sp];
    }
    return w;
}

static bool inside(const Aabb& b, const double* p, double tol) {
    for (int k = 0; k < 3; ++k)
        if (p[k] < b.lo[k] - tol || p[k] > b.hi[k] + tol) return false;
    return true;
}

// the tree's structure and, for every triangle, the leaves that reference it
static bool check_tree(const Bvh2& tree, uint32_t n, std::vector<std::vector<uint32_t>>* leaves_of, uint64_t* refs) {
    std::vector<uint32_t> st{tree.root};
    uint64_t interior = 0, prims = 0;
    while (!st.empty()) {
        const uint32_t ni = st.back();
        st.pop_back();
        const Bvh2Node& nd = tree.nodes[ni];
        if (nd.count > 0) {
            if (nd.n_interior != 0 || nd.n_prims != nd.count || (size_t)nd.first + nd.count > tree.order.size()) return false;
            for (uint32_t k = 0; k < nd.count; ++k) {
                const uint32_t p = tree.order[nd.first + k];
                if (p >= n) return false;
                (*leaves_of)[p].push_back(ni);
            }
            prims += nd.count;
        } else {
            const Bvh2Node &l = tree.nodes[nd.left], &r = tree.nodes[nd.right];
            if (nd.n_interior != 1 + l.n_interior + r.n_interior || nd.n_prims != l.n_prims + r.n_prims) return false;
            for (int a = 0; a < 3; ++a)
                if (l.box.lo[a] < nd.box.lo[a] || l.box.hi[a] > nd.box.hi[a] || r.box.lo[a] < nd.box.lo[a] || r.box.hi[a] > nd.box.hi[a])
                    return false;
            ++interior;
            st.push_back((uint32_t)nd.left);
            st.push_back((uint32_t)nd.right);
        }
    }
    *refs = prims;
    return prims == tree.order.size() && prims == tree.nodes[tree.root].n_prims && interior == tree.nodes[tree.root].n_interior &&
           tree.nodes.size() == 2 * interior + 1;
}

// a fingerprint of the tree that does not depend on node numbering or on the order of references inside a leaf
static uint64_t fingerprint(const Bvh2& tree, uint32_t ni) {
    const Bvh2Node& nd = tree.nodes[ni];
    uint64_t h = 1469598103934665603ull;
    auto mix = [&h](uint64_t x) { h = (h ^ x) * 1099511628211ull; };
    for (int k = 0; k < 3; ++k) {
        uint64_t a, b;
        memcpy(&a, &nd.box.lo[k], 8);
        memcpy(&b, &nd.box.hi[k], 8);
        mix(a);
        mix(b);
    }
    if (nd.count > 0) {
        std::vector<uint32_t> ids(tree.order.begin() + nd.first, tree.order.begin() + nd.first + nd.count);
        std::sort(ids.begin(), ids.end());
        for (uint32_t id : ids) mix(id);
        return h;
    }
    mix(fingerprint(tree, (uint32_t)nd.left));
    mix(fingerprint(tree, (uint32_t)nd.right));
    return h;
}

template <class F>
static void parallel_for(size_t n, F&& f) {
    const int th = std::max(1u, std::thread::hardware_concurrency());
    std::vector<std::thread> ts;
    for (int t = 0; t < th; ++t) ts.emplace_back([&, t] {
        for (size_t i = t; i < n; i += th) f(i);
    });
    for (auto& t : ts) t.join();
}

int main(int argc, char** argv) {
    if (argc < 3) {
        fprintf(stderr, "usage: sbvh_check TRIS RAYS [n_rays]\n");
        return 3;
    }
    const std::vector<double> tris = read_f64(argv[1]);
    const std::vector<double> rays = read_f64(argv[2]);
    const uint32_t n = (uint32_t)(tris.size() / 9);
    size_t n_rays = rays.size() / 7;
    if (argc > 3) n_rays = std::min(n_rays, (size_t)atoll(argv[3]));
    std::vector<Aabb> boxes(n);
    Aabb world;
    for (uint32_t i = 0; i < n; ++i) {
        for (int v = 0; v < 3; ++v) boxes[i].grow(&tris[9 * (size_t)i + 3 * v]);
        world.grow(boxes[i]);
    }
    SahParams prm;
    prm.max_leaf = 4;  // what the commit passes for max_prims_in_node = 0
    if (getenv("T")) prm.n_threads = atoi(getenv("T"));
    if (getenv("RRT_SAH_CI")) prm.cost_intersect = atof(getenv("RRT_SAH_CI"));
    if (getenv("RRT_SBVH_ALPHA")) prm.split_alpha = atof(getenv("RRT_SBVH_ALPHA"));
    if (getenv("RRT_SBVH_CAP")) prm.split_cap = atof(getenv("RRT_SBVH_CAP"));
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };

    Bvh2 obj, spl;
    double t0 = now();
    build_sah(AabbSpan(boxes), prm, &obj);
    double t1 = now();
    SplitTriangles st;
    st.verts = tris.data();
    build_sah(AabbSpan(boxes), st, prm, &spl);
    double t2 = now();
    printf("params alpha=%g cap=%g ci=%g threads=%d\n", prm.split_alpha, prm.split_cap, prm.cost_intersect, prm.n_threads);
    printf("object  build %.3f s: %zu nodes, %u leaves, %zu refs, depth %u\n", t1 - t0, obj.nodes.size(), obj.n_leaves, obj.order.size(), obj.max_depth);
    printf("spatial build %.3f s: %zu nodes, %u leaves, %zu refs (%.4f n), depth %u\n", t2 - t1, spl.nodes.size(), spl.n_leaves,
           spl.order.size(), (double)spl.order.size() / n, spl.max_depth);
    printf("fingerprint %016llx refs %zu depth %u\n", (unsigned long long)fingerprint(spl, spl.root), spl.order.size(), spl.max_depth);

    // ---- the spatial tree is a valid tree over every point of every triangle ----
    std::vector<std::vector<uint32_t>> leaves_of(n);
    uint64_t refs = 0;
    bool ok = check_tree(spl, n, &leaves_of, &refs);
    printf("structure %s\n", ok ? "VALID" : "BROKEN");
    if (!ok) return 2;
    double scale = 0.0;
    for (int k = 0; k < 3; ++k) scale = std::max(scale, std::max(std::fabs(world.lo[k]), std::fabs(world.hi[k])));
    // (the packer pads every box outward by scale * 2^-19: a crossing point's f64 rounding is 7 orders below that)
    const double tol = scale * 1e-12;
    static const double kBary[][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}, {0.5, 0.5, 0}, {0, 0.5, 0.5}, {0.5, 0, 0.5},
                                      {0.25, 0.75, 0}, {0, 0.1, 0.9}, {0.7, 0, 0.3}, {1.0 / 3, 1.0 / 3, 1.0 / 3},
                                      {0.6, 0.3, 0.1}, {0.05, 0.15, 0.8}, {0.2, 0.6, 0.2}, {0.45, 0.1, 0.45}};
    std::vector<uint8_t> bad(n, 0);
    parallel_for(n, [&](size_t i) {
        if (leaves_of[i].empty()) {
            bad[i] = 1;
            return;
        }
        const double* v = &tris[9 * i];
        for (const auto& b : kBary) {
            double p[3];
            for (int k = 0; k < 3; ++k) p[k] = b[0] * v[k] + b[1] * v[3 + k] + b[2] * v[6 + k];
            bool in = false;
            for (uint32_t li : leaves_of[i]) in = in || inside(spl.nodes[li].box, p, tol);
            if (!in) bad[i] = 2;
        }
    });
    size_t unreferenced = 0, uncovered = 0;
    for (uint32_t i = 0; i < n; ++i) {
        unreferenced += bad[i] == 1;
        uncovered += bad[i] == 2;
    }
    printf("coverage %s: %zu unreferenced triangles, %zu with a sampled point outside their leaves\n",
           unreferenced + uncovered == 0 ? "COMPLETE" : "INCOMPLETE", unreferenced, uncovered);
    if (unreferenced + uncovered) return 2;

    // ---- the two trees give the same closest hits; what each walk costs ----
    std::vector<Walk> wo(n_rays), ws(n_rays);
    parallel_for(n_rays, [&](size_t i) {
        wo[i] = closest(obj, tris.data(), &rays[7 * i]);
        ws[i] = closest(spl, tris.data(), &rays[7 * i]);
    });
    size_t differ = 0, hits = 0;
    double vo = 0, to = 0, vs = 0, ts = 0;
    for (size_t i = 0; i < n_rays; ++i) {
        uint64_t a, b;
        memcpy(&a, &wo[i].t, 8);
        memcpy(&b, &ws[i].t, 8);
        differ += wo[i].prim != ws[i].prim || a != b;
        hits += wo[i].prim != 0xFFFFFFFFu;
        vo += wo[i].visits;
        to += wo[i].tests;
        vs += ws[i].visits;
        ts += ws[i].tests;
    }
    printf("rays %zu, %zu hit: closest hits %s (%zu differ)\n", n_rays, hits, differ == 0 ? "IDENTICAL" : "DIFFERENT", differ);
    printf("cost object  : %.2f interior visits, %.2f leaf tests per ray\n", vo / n_rays, to / n_rays);
    printf("cost spatial : %.2f interior visits, %.2f leaf tests per ray\n", vs / n_rays, ts / n_rays);
    return differ == 0 ? 0 : 1;
}

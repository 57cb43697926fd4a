#include "bvh_sah.hpp"

#include <algorithm>
#include <atomic>
#include <future>
#include <thread>

namespace rrt {
namespace {

constexpr int kBins = 16;

inline double half_area(const Aabb& b) {
    if (b.empty()) return 0.0;
    double dx = b.hi[0] - b.lo[0], dy = b.hi[1] - b.lo[1], dz = b.hi[2] - b.lo[2];
    return dx * dy + dx * dz + dy * dz;
}

// Branch-free box growth: minsd / maxsd and an unconditional store.  (Aabb::grow's `if (p < lo) lo = p` compiles to a
// conditional store behind a branch, and the bins of a SAH pass are as unpredictable as branches get: the binning loop
// spent 155 cycles per primitive on them.)
inline void grow_box(Aabb& a, const Aabb& b) {
    for (int k = 0; k < 3; ++k) {
        a.lo[k] = std::min(a.lo[k], b.lo[k]);
        a.hi[k] = std::max(a.hi[k], b.hi[k]);
    }
}
template <class T>
inline void grow_point(Aabb& a, const T c[3]) {
    for (int k = 0; k < 3; ++k) {
        a.lo[k] = std::min(a.lo[k], (double)c[k]);
        a.hi[k] = std::max(a.hi[k], (double)c[k]);
    }
}

// The bins of one node: for every axis, the boxes and counts of the primitives whose centroid falls into each of kBins
// slices of the node's centroid box.  ONE pass over the node's primitives fills all three axes; the bins of the chosen
// axis also give both children their boxes and the partition pass their centroid boxes, so a child does not walk its
// primitives to find them.
struct Bins {
    Aabb box[3][kBins];
    uint32_t cnt[3][kBins];
    Bins() {
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < kBins; ++b) cnt[a][b] = 0;
    }
    void merge(const Bins& o) {
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < kBins; ++b) {
                grow_box(box[a][b], o.box[a][b]);
                cnt[a][b] += o.cnt[a][b];
            }
    }
};

// The bins of a spatial split (SBVH): for every axis, kBins equal slabs of the node's box.  A reference enters the slab
// holding its box's low side and exits the one holding its high side; a triangle adds to each slab in between the box of
// its part inside that slab.  A reference that cannot be split (a sphere) enters and exits its centroid's slab whole.
struct SpatialBins {
    Aabb box[3][kBins];
    uint32_t enter[3][kBins], exit[3][kBins];
    SpatialBins() {
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < kBins; ++b) enter[a][b] = exit[a][b] = 0;
    }
    void merge(const SpatialBins& o) {
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < kBins; ++b) {
                grow_box(box[a][b], o.box[a][b]);
                enter[a][b] += o.enter[a][b];
                exit[a][b] += o.exit[a][b];
            }
    }
};

// The box of the part of triangle v[0..8] with slo <= x[axis] <= shi, cut down to `ref` (the reference's box, which
// ancestors' splits may already have clipped): vertices inside the slab and the points where edges cross its planes.
// Empty when nothing of the triangle lies in both.  (A crossing point's other coordinates carry f64 rounding, far
// below the packer's outward padding of every box.)
inline Aabb clip_triangle(const double* v, int axis, double slo, double shi, const Aabb& ref) {
    Aabb out;
    for (int e = 0; e < 3; ++e) {
        const double* a = v + 3 * e;
        const double* b = v + 3 * ((e + 1) % 3);
        const double pa = a[axis], pb = b[axis];
        if (pa >= slo && pa <= shi) grow_point(out, a);
        for (const double plane : {slo, shi}) {
            if ((pa < plane && pb > plane) || (pa > plane && pb < plane)) {
                const double t = (plane - pa) / (pb - pa);
                double p[3];
                for (int k = 0; k < 3; ++k) p[k] = a[k] + t * (b[k] - a[k]);
                p[axis] = plane;
                grow_point(out, p);
            }
        }
    }
    for (int k = 0; k < 3; ++k) {
        out.lo[k] = std::max(out.lo[k], ref.lo[k]);
        out.hi[k] = std::min(out.hi[k], ref.hi[k]);
        if (!(out.lo[k] <= out.hi[k])) return Aabb();
    }
    return out;
}

// What the builder moves around: a reference's box, its centroid (fp32 is plenty for binning) and its primitive's index,
// 64 bytes.  A node's references are a contiguous run of these, partitioned in place — every pass of every level streams
// through memory instead of gathering 48-byte boxes through an index array (which is what a 4 Mi-primitive build spent
// its time on).  With spatial splits a node's run is followed by free slots (its share of the reference budget) that
// its subtree may fill with duplicated references.
struct Item {
    Aabb box;
    float c[3];
    uint32_t id;
    void set_box(const Aabb& b) {
        box = b;
        for (int k = 0; k < 3; ++k) c[k] = (float)(0.5 * (b.lo[k] + b.hi[k]));
    }
};
struct Builder {
    SahParams prm;
    RawBuf<Item> items, scratch;  // scratch: the large nodes' parallel partition
    std::vector<Bvh2Node, NoInitAlloc<Bvh2Node>> nodes;
    std::atomic<uint32_t> next_node{0};
    std::atomic<int> active{1};
    std::atomic<uint32_t> n_leaves{0};
    int max_threads = 1;
    uint32_t n_total = 0;
    // spatial splits: the triangles' vertices (9 doubles per primitive; null = object splits only), which primitives are
    // triangles (null = all), and the overlap (split_alpha x the root's half area) above which a node tries one
    const double* tv = nullptr;
    const uint8_t* tmask = nullptr;
    double alpha_area = 0.0;
    bool is_tri(uint32_t id) const { return tmask == nullptr || tmask[id] != 0; }
    static constexpr uint32_t kParallelNode = 1u << 18;  // nodes of at least this many primitives split their passes over threads
    // nodes of fewer references do not try spatial splits: on the config-3 / config-5 soups the budget is spent near the
    // top, and below this the search costs build time without changing the walk (63.01 vs 63.05 visits per ray on
    // config 3, profiles/r3_sbvh_sweep.txt)
    static constexpr uint32_t kSpatialMinRefs = 512;

    Builder(size_t n, size_t n_scratch, const SahParams& p) : prm(p), items(n), scratch(n_scratch) {}

    uint32_t make_leaf(uint32_t ni, uint32_t begin, uint32_t end) {
        nodes[ni].first = begin;
        nodes[ni].count = end - begin;
        nodes[ni].left = nodes[ni].right = -1;
        nodes[ni].n_interior = 0;
        nodes[ni].n_prims = end - begin;
        n_leaves.fetch_add(1, std::memory_order_relaxed);
        return 1;  // depth of the subtree, in nodes
    }

    // threads a node of n primitives may use for its own passes: its share of the machine (the top of the tree is a handful
    // of huge nodes — one thread each would leave the others idle for most of the build)
    int node_threads(uint32_t n) const {
        if (n < kParallelNode || max_threads <= 1) return 1;
        const uint64_t t = ((uint64_t)max_threads * n + n_total - 1) / n_total;
        return (int)std::min<uint64_t>(std::max<uint64_t>(t, 1), (uint64_t)max_threads);
    }
    template <class F>
    static void for_chunks(uint32_t begin, uint32_t end, int threads, F&& f) {  // f(chunk index, chunk begin, chunk end)
        if (threads <= 1) {
            f(0, begin, end);
            return;
        }
        const uint32_t per = (end - begin + threads - 1) / threads;
        std::vector<std::future<void>> futs;
        for (int t = 1; t < threads; ++t) {
            const uint32_t b = std::min(end, begin + (uint32_t)t * per), e = std::min(end, b + per);
            futs.push_back(std::async(std::launch::async, [&f, t, b, e] { f(t, b, e); }));
        }
        f(0, begin, std::min(end, begin + per));
        for (auto& fu : futs) fu.get();
    }

    void bounds(uint32_t begin, uint32_t end, Aabb* box, Aabb* cbox) {
        const int threads = node_threads(end - begin);
        std::vector<Aabb> pb(threads), pc(threads);
        for_chunks(begin, end, threads, [&](int t, uint32_t b, uint32_t e) {
            Aabb bb, cc;
            for (uint32_t i = b; i < e; ++i) {
                grow_box(bb, items[i].box);
                grow_point(cc, items[i].c);
            }
            pb[t] = bb;
            pc[t] = cc;
        });
        for (int t = 0; t < threads; ++t) {
            box->grow(pb[t]);
            cbox->grow(pc[t]);
        }
    }

    // The slabs of a spatial split over a node's box, and which of them a coordinate falls into.  Binning and partition
    // both decide with bin(), so a reference goes to the sides the bins counted it on (or, clipped to nothing on one, to
    // fewer).
    struct SlabGrid {
        double lo[3], w[3], scale[3];
        int bin(int axis, double x) const {
            int k = (int)((x - lo[axis]) * scale[axis]);
            return k < 0 ? 0 : (k >= kBins ? kBins - 1 : k);
        }
    };
    struct SpatialChoice {
        int axis = -1, split = -1;
        double cost = INFINITY;
        SlabGrid g;
    };
    // SBVH's spatial split search: the cheapest plane on a slab boundary whose duplicated references fit the node's free
    // slots and that leaves each side with fewer references than the node
    SpatialChoice find_spatial(uint32_t begin, uint32_t end, uint32_t slack, const Aabb& box, int threads) {
        SpatialChoice ch;
        SlabGrid& g = ch.g;
        bool live[3];
        for (int axis = 0; axis < 3; ++axis) {
            const double ext = box.hi[axis] - box.lo[axis];
            live[axis] = ext > 0.0;
            g.lo[axis] = box.lo[axis];
            g.w[axis] = ext / kBins;
            g.scale[axis] = live[axis] ? kBins / ext : 0.0;
        }
        SpatialBins bins;
        std::vector<SpatialBins> part(threads > 1 ? threads - 1 : 0);
        for_chunks(begin, end, threads, [&](int t, uint32_t b, uint32_t e) {
            SpatialBins& B = t == 0 ? bins : part[t - 1];
            for (uint32_t i = b; i < e; ++i) {
                const Item& it = items[i];
                for (int axis = 0; axis < 3; ++axis) {
                    if (!live[axis]) continue;
                    if (!is_tri(it.id)) {
                        const int k = g.bin(axis, it.c[axis]);
                        B.enter[axis][k]++;
                        B.exit[axis][k]++;
                        grow_box(B.box[axis][k], it.box);
                        continue;
                    }
                    const int b0 = g.bin(axis, it.box.lo[axis]), b1 = g.bin(axis, it.box.hi[axis]);
                    B.enter[axis][b0]++;
                    B.exit[axis][b1]++;
                    if (b0 == b1) {
                        grow_box(B.box[axis][b0], it.box);
                        continue;
                    }
                    const double* v = tv + 9 * (size_t)it.id;
                    for (int k = b0; k <= b1; ++k) {
                        const double slo = k == b0 ? -INFINITY : g.lo[axis] + k * g.w[axis];
                        const double shi = k == b1 ? INFINITY : g.lo[axis] + (k + 1) * g.w[axis];
                        const Aabb c = clip_triangle(v, axis, slo, shi, it.box);
                        if (!c.empty()) grow_box(B.box[axis][k], c);
                    }
                }
            }
        });
        for (const SpatialBins& o : part) bins.merge(o);
        const uint32_t n = end - begin;
        for (int axis = 0; axis < 3; ++axis) {
            if (!live[axis]) continue;
            double right_area[kBins];
            uint32_t right_cnt[kBins];
            Aabb acc;
            uint32_t cnt = 0;
            for (int b = kBins - 1; b > 0; --b) {
                grow_box(acc, bins.box[axis][b]);
                cnt += bins.exit[axis][b];
                right_area[b] = half_area(acc);
                right_cnt[b] = cnt;
            }
            acc = Aabb();
            cnt = 0;
            for (int b = 0; b < kBins - 1; ++b) {
                grow_box(acc, bins.box[axis][b]);
                cnt += bins.enter[axis][b];
                const uint32_t rc = right_cnt[b + 1];
                if (cnt == 0 || rc == 0 || cnt >= n || rc >= n || (uint64_t)cnt + rc > (uint64_t)n + slack) continue;
                const double cost = half_area(acc) * cnt + right_area[b + 1] * rc;
                if (cost < ch.cost) {
                    ch.cost = cost;
                    ch.axis = axis;
                    ch.split = b;
                }
            }
        }
        return ch;
    }

    // Moves the node's references to the two sides of a spatial split: a triangle that crosses the plane goes to both, with
    // the box of its part on each side.  Each chunk of threads keeps its own runs, and the runs are laid out in chunk
    // order, so the result does not depend on the thread count.  The left run starts at `begin`, the right one after the
    // left's share of the free slots that are left.
    void spatial_partition(uint32_t begin, uint32_t end, uint32_t cap, const SpatialChoice& sp, int threads, uint32_t* l_end,
                           uint32_t* r_begin, uint32_t* r_end, Aabb* lbox, Aabb* lcbox, Aabb* rbox, Aabb* rcbox) {
        struct Sides {
            std::vector<Item> l, r;
            Aabb lb, lc, rb, rc;
        };
        std::vector<Sides> sides(threads);
        const int axis = sp.axis, split = sp.split;
        const double pos = sp.g.lo[axis] + (split + 1) * sp.g.w[axis];
        for_chunks(begin, end, threads, [&](int t, uint32_t b, uint32_t e) {
            Sides& S = sides[t];
            auto left = [&](const Item& it) {
                S.l.push_back(it);
                grow_box(S.lb, it.box);
                grow_point(S.lc, it.c);
            };
            auto right = [&](const Item& it) {
                S.r.push_back(it);
                grow_box(S.rb, it.box);
                grow_point(S.rc, it.c);
            };
            for (uint32_t i = b; i < e; ++i) {
                const Item& it = items[i];
                if (!is_tri(it.id)) {
                    if (sp.g.bin(axis, it.c[axis]) <= split) left(it); else right(it);
                    continue;
                }
                if (sp.g.bin(axis, it.box.hi[axis]) <= split) {
                    left(it);
                } else if (sp.g.bin(axis, it.box.lo[axis]) > split) {
                    right(it);
                } else {
                    const double* v = tv + 9 * (size_t)it.id;
                    const Aabb lb = clip_triangle(v, axis, -INFINITY, pos, it.box), rb = clip_triangle(v, axis, pos, INFINITY, it.box);
                    if (lb.empty() && rb.empty()) {  // (only rounding can lose both parts: keep the reference whole)
                        if (it.c[axis] <= pos) left(it); else right(it);
                        continue;
                    }
                    Item c = it;
                    if (!lb.empty()) {
                        c.set_box(lb);
                        left(c);
                    }
                    if (!rb.empty()) {
                        c.set_box(rb);
                        right(c);
                    }
                }
            }
        });
        uint64_t n_l = 0, n_r = 0;
        for (const Sides& S : sides) {
            n_l += S.l.size();
            n_r += S.r.size();
            grow_box(*lbox, S.lb);
            grow_box(*lcbox, S.lc);
            grow_box(*rbox, S.rb);
            grow_box(*rcbox, S.rc);
        }
        // (find_spatial counted at least as many references on each side, and kept their total within the free slots)
        const uint64_t free_slots = (uint64_t)(cap - begin) - n_l - n_r;
        const uint32_t slack_l = (uint32_t)(free_slots * n_l / (n_l + n_r));
        uint32_t at = begin;
        for (const Sides& S : sides) at = (uint32_t)(std::copy(S.l.begin(), S.l.end(), items.get() + at) - items.get());
        *l_end = at;
        *r_begin = at = at + slack_l;
        for (const Sides& S : sides) at = (uint32_t)(std::copy(S.r.begin(), S.r.end(), items.get() + at) - items.get());
        *r_end = at;
    }

    // `box` / `cbox`: the node's box and centroid box when the parent's bins gave them, else null (the root; children of a
    // median split).  [end, cap): the node's free slots, which duplicated references of its subtree may take.
    // returns the depth of the subtree it built (the traversal stack is sized from it)
    uint32_t build(uint32_t ni, uint32_t begin, uint32_t end, uint32_t cap, const Aabb* box_in, const Aabb* cbox_in) {
        const uint32_t n = end - begin;
        Aabb box, cbox;
        if (box_in) {
            box = *box_in;
            cbox = *cbox_in;
        } else {
            bounds(begin, end, &box, &cbox);
        }
        nodes[ni].box = box;
        if (n == 1) return make_leaf(ni, begin, end);

        // binned SAH over all three axes, one pass
        double lo[3], scale[3];
        bool live[3];
        for (int axis = 0; axis < 3; ++axis) {
            const double ext = cbox.hi[axis] - cbox.lo[axis];
            lo[axis] = cbox.lo[axis];
            live[axis] = ext > 0.0;
            scale[axis] = live[axis] ? kBins / ext : 0.0;
        }
        const int threads = node_threads(n);
        Bins bins;                               // (on the stack: two million nodes do not each want a heap allocation)
        std::vector<Bins> part(threads > 1 ? threads - 1 : 0);
        for_chunks(begin, end, threads, [&](int t, uint32_t b, uint32_t e) {
            Bins& B = t == 0 ? bins : part[t - 1];
            for (uint32_t i = b; i < e; ++i) {
                const Item& it = items[i];
                for (int axis = 0; axis < 3; ++axis) {
                    if (!live[axis]) continue;
                    int k = (int)((it.c[axis] - lo[axis]) * scale[axis]);
                    k = k < 0 ? 0 : (k >= kBins ? kBins - 1 : k);
                    B.cnt[axis][k]++;
                    grow_box(B.box[axis][k], it.box);
                }
            }
        });
        for (const Bins& o : part) bins.merge(o);

        double best_cost = INFINITY;
        int best_axis = -1, best_split = -1;
        const double parent_area = half_area(box);
        for (int axis = 0; axis < 3; ++axis) {
            if (!live[axis]) continue;
            double right_area[kBins];
            uint32_t right_cnt[kBins];
            Aabb acc;
            uint32_t cnt = 0;
            for (int b = kBins - 1; b > 0; --b) {
                grow_box(acc, bins.box[axis][b]);
                cnt += bins.cnt[axis][b];
                right_area[b] = half_area(acc);
                right_cnt[b] = cnt;
            }
            acc = Aabb();
            cnt = 0;
            for (int b = 0; b < kBins - 1; ++b) {
                grow_box(acc, bins.box[axis][b]);
                cnt += bins.cnt[axis][b];
                if (cnt == 0 || right_cnt[b + 1] == 0) continue;
                double cost = half_area(acc) * cnt + right_area[b + 1] * right_cnt[b + 1];
                if (cost < best_cost) {
                    best_cost = cost;
                    best_axis = axis;
                    best_split = b;
                }
            }
        }
        uint32_t mid = begin;
        bool child_boxes = false, spatial = false;
        Aabb lbox, lcbox, rbox, rcbox;
        uint32_t l_end = 0, r_begin = 0, r_end = 0;  // the children: [begin, l_end) and [r_begin, r_end)
        if (best_axis < 0) {
            // all centroids coincide: nothing to bin on
            if (n <= prm.max_leaf) return make_leaf(ni, begin, end);
            mid = begin + n / 2;
        } else {
            // a spatial split is worth its binning pass only where the object split leaves the children overlapping
            SpatialChoice sp;
            if (tv != nullptr && end < cap && n >= kSpatialMinRefs) {
                Aabb ol, orr;
                for (int b = 0; b < kBins; ++b) grow_box(b <= best_split ? ol : orr, bins.box[best_axis][b]);
                Aabb ov;
                bool overlap = true;
                for (int k = 0; k < 3; ++k) {
                    ov.lo[k] = std::max(ol.lo[k], orr.lo[k]);
                    ov.hi[k] = std::min(ol.hi[k], orr.hi[k]);
                    overlap = overlap && ov.lo[k] <= ov.hi[k];
                }
                if (overlap && half_area(ov) > alpha_area) sp = find_spatial(begin, end, cap - end, box, threads);
            }
            const double cost = std::min(best_cost, sp.cost);
            double split_cost = prm.cost_traverse + prm.cost_intersect * cost / (parent_area > 0 ? parent_area : 1.0);
            double leaf_cost = prm.cost_intersect * n;
            if (n <= prm.max_leaf && leaf_cost <= split_cost) return make_leaf(ni, begin, end);
            if (sp.cost < best_cost) {
                spatial_partition(begin, end, cap, sp, threads, &l_end, &r_begin, &r_end, &lbox, &lcbox, &rbox, &rcbox);
                spatial = child_boxes = true;
            } else {
                const double plo = lo[best_axis], pscale = scale[best_axis];
                auto goes_left = [&](const Item& it) {
                    int b = (int)((it.c[best_axis] - plo) * pscale);
                    b = b < 0 ? 0 : (b >= kBins ? kBins - 1 : b);
                    return b <= best_split;
                };
                uint32_t n_left = 0;
                for (int b = 0; b <= best_split; ++b) n_left += bins.cnt[best_axis][b];
                if (threads > 1) {
                    // stable two-sided scatter through the scratch array: every chunk knows where its left and right runs go
                    std::vector<uint32_t> lefts(threads, 0);
                    for_chunks(begin, end, threads, [&](int t, uint32_t b, uint32_t e) {
                        uint32_t c = 0;
                        for (uint32_t i = b; i < e; ++i) c += goes_left(items[i]) ? 1u : 0u;
                        lefts[t] = c;
                    });
                    std::vector<uint32_t> lpos(threads), rpos(threads);
                    const uint32_t per = (n + threads - 1) / threads;
                    uint32_t lacc = begin, racc = begin + n_left;
                    for (int t = 0; t < threads; ++t) {
                        const uint32_t b = std::min(end, begin + (uint32_t)t * per), e = std::min(end, b + per);
                        lpos[t] = lacc;
                        rpos[t] = racc;
                        lacc += lefts[t];
                        racc += (e - b) - lefts[t];
                    }
                    std::vector<Aabb> plc(threads), prc(threads);
                    for_chunks(begin, end, threads, [&](int t, uint32_t b, uint32_t e) {
                        uint32_t l = lpos[t], r = rpos[t];
                        Aabb lc, rc;
                        for (uint32_t i = b; i < e; ++i) {
                            const Item& it = items[i];
                            if (goes_left(it)) {
                                scratch[l++] = it;
                                grow_point(lc, it.c);
                            } else {
                                scratch[r++] = it;
                                grow_point(rc, it.c);
                            }
                        }
                        plc[t] = lc;
                        prc[t] = rc;
                    });
                    for (int t = 0; t < threads; ++t) {
                        grow_box(lcbox, plc[t]);
                        grow_box(rcbox, prc[t]);
                    }
                    for_chunks(begin, end, threads, [&](int, uint32_t b, uint32_t e) {
                        std::copy(scratch.get() + b, scratch.get() + e, items.get() + b);
                    });
                    mid = begin + n_left;
                } else {
                    // two-pointer partition that looks at every primitive exactly once (and so can grow both sides' centroid boxes)
                    Item *lp = items.get() + begin, *rp = items.get() + end;
                    for (;;) {
                        while (lp < rp && goes_left(*lp)) {
                            grow_point(lcbox, lp->c);
                            ++lp;
                        }
                        while (lp < rp && !goes_left(*(rp - 1))) {
                            --rp;
                            grow_point(rcbox, rp->c);
                        }
                        if (rp - lp < 2) break;  // lp == rp (an item at lp == rp - 1 was decided by one of the loops)
                        // *lp goes right, *(rp - 1) goes left: swap them, each is now decided
                        std::swap(*lp, *(rp - 1));
                        grow_point(lcbox, lp->c);
                        ++lp;
                        --rp;
                        grow_point(rcbox, rp->c);
                    }
                    mid = (uint32_t)(lp - items.get());
                }
                if (mid == begin || mid == end) {
                    mid = begin + n / 2;
                } else {
                    child_boxes = true;
                    for (int b = 0; b < kBins; ++b) grow_box(b <= best_split ? lbox : rbox, bins.box[best_axis][b]);
                }
            }
        }
        if (!spatial) {
            // object (or median) split: [begin, mid) | [mid, end); the right run moves up past the left's share of the
            // free slots
            const uint32_t slack_l = (uint32_t)((uint64_t)(cap - end) * (mid - begin) / n);
            if (slack_l > 0) std::copy_backward(items.get() + mid, items.get() + end, items.get() + end + slack_l);
            l_end = mid;
            r_begin = mid + slack_l;
            r_end = end + slack_l;
        }
        uint32_t l = next_node.fetch_add(2, std::memory_order_relaxed);
        uint32_t r = l + 1;
        nodes[ni].left = (int32_t)l;
        nodes[ni].right = (int32_t)r;
        nodes[ni].first = 0;
        nodes[ni].count = 0;
        const Aabb *lb = child_boxes ? &lbox : nullptr, *lc = child_boxes ? &lcbox : nullptr;
        const Aabb *rb = child_boxes ? &rbox : nullptr, *rc = child_boxes ? &rcbox : nullptr;
        const uint32_t par_min = 1u << 12;
        uint32_t dl, dr;
        if (n >= par_min && active.load(std::memory_order_relaxed) < max_threads) {
            active.fetch_add(1);
            auto fut = std::async(std::launch::async, [this, l, begin, l_end, r_begin, lb, lc] {
                const uint32_t d = build(l, begin, l_end, r_begin, lb, lc);
                active.fetch_sub(1);
                return d;
            });
            dr = build(r, r_begin, r_end, cap, rb, rc);
            dl = fut.get();
        } else {
            dl = build(l, begin, l_end, r_begin, lb, lc);
            dr = build(r, r_begin, r_end, cap, rb, rc);
        }
        nodes[ni].n_interior = 1 + nodes[l].n_interior + nodes[r].n_interior;
        nodes[ni].n_prims = nodes[l].n_prims + nodes[r].n_prims;  // the leaves' references: n, plus the subtree's duplicates
        return 1 + std::max(dl, dr);
    }
};

}  // namespace

namespace {

void build_tree(AabbSpan boxes, const SplitTriangles* tris, const SahParams& params, Bvh2* out) {
    const uint32_t n = (uint32_t)boxes.size();
    int max_threads = params.n_threads > 0 ? params.n_threads : (int)std::thread::hardware_concurrency();
    if (max_threads < 1) max_threads = 1;
    const bool parallel_nodes = n >= Builder::kParallelNode && max_threads > 1;
    // the reference budget: free slots for the duplicates of spatial splits, shared out down the tree
    const double extra = tris != nullptr && tris->verts != nullptr ? std::max(0.0, params.split_cap - 1.0) : 0.0;
    const uint32_t n_cap = (uint32_t)std::min<double>((double)n + std::floor(extra * n), (double)(1u << 28));
    Builder b(n_cap, parallel_nodes ? n_cap : 0, params);
    if (b.prm.max_leaf < 1) b.prm.max_leaf = 1;
    if (b.prm.max_leaf > 8) b.prm.max_leaf = 8;
    b.max_threads = max_threads;
    b.n_total = n;
    Builder::for_chunks(0, n, parallel_nodes ? max_threads : 1, [&](int, uint32_t lo, uint32_t hi) {
        for (uint32_t i = lo; i < hi; ++i) {
            Item& it = b.items[i];
            it.box = boxes[i];
            for (int k = 0; k < 3; ++k) it.c[k] = (float)(0.5 * (boxes[i].lo[k] + boxes[i].hi[k]));
            it.id = i;
        }
    });
    b.nodes.resize(2 * (size_t)n_cap + 1);
    b.next_node = 1;
    uint32_t depth;
    if (n_cap > n) {
        b.tv = tris->verts;
        b.tmask = tris->is_tri;
        Aabb box, cbox;
        b.bounds(0, n, &box, &cbox);
        b.alpha_area = params.split_alpha * half_area(box);
        depth = b.build(0, 0, n, n_cap, &box, &cbox);
    } else {
        depth = b.build(0, 0, n, n, nullptr, nullptr);
    }
    b.nodes.resize(b.next_node.load());
    const uint32_t n_refs = b.nodes[0].n_prims;
    out->order.resize(n_refs);
    if (n_cap > n) {
        // close the free slots the subtrees left: leaf ranges are disjoint runs of the item array, in item order
        std::vector<uint32_t> at(n_cap + 1, 0);
        for (const Bvh2Node& nd : b.nodes)
            for (uint32_t k = 0; k < nd.count; ++k) at[nd.first + k] = 1;
        uint32_t acc = 0;
        for (uint32_t i = 0; i <= n_cap; ++i) {
            const uint32_t used = at[i];
            at[i] = acc;
            if (i < n_cap && used) out->order[acc++] = b.items[i].id;
        }
        for (Bvh2Node& nd : b.nodes)
            if (nd.count > 0) nd.first = at[nd.first];
    } else {
        Builder::for_chunks(0, n, parallel_nodes ? max_threads : 1, [&](int, uint32_t lo, uint32_t hi) {
            for (uint32_t i = lo; i < hi; ++i) out->order[i] = b.items[i].id;
        });
    }
    out->nodes = std::move(b.nodes);
    out->root = 0;
    out->n_leaves = b.n_leaves.load();
    out->max_depth = depth;
}

}  // namespace

void build_sah(AabbSpan boxes, const SahParams& params, Bvh2* out) { build_tree(boxes, nullptr, params, out); }

void build_sah(AabbSpan boxes, const SplitTriangles& tris, const SahParams& params, Bvh2* out) {
    build_tree(boxes, &tris, params, out);
}

}  // namespace rrt

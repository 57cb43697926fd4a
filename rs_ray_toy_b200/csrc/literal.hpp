// The LITERAL parity tier on the device (RRT_BUILD_LITERAL): the reference's own HLBVH
// (bvh_hlbvh.cpp), walked in the reference's order with the reference's accept rules in f64 —
// BVHAccel::intersect / intersect_p (src/bvh.rs:123-236) as they are, quirks included
// (SURVEY.md Appendix A: Q1-Q6, Q9).  One thread per ray; this tier exists to reproduce the
// reference bit for bit on its own scenes (config 1), not for throughput.
#pragma once
#include <string>
#include <vector>

#include "aggregate.hpp"

namespace rrt {

struct ShadeScene;

class LiteralAggregate : public RayTracer {
  public:
    LiteralAggregate() = default;
    ~LiteralAggregate() override;
    int build(int device, const HostScene& scene, uint32_t max_prims_in_node, std::string* err);
    int closest_hit(uint64_t n, const rrt_ray* d_rays, rrt_hit* d_hits, void* stream, std::string* err,
                    int* launches = nullptr) const override;
    int any_hit(uint64_t n, const rrt_ray* d_rays, uint8_t* d_occluded, void* stream, std::string* err,
                int* launches = nullptr) const override;
    int closest_hit_indirect(uint64_t capacity, const uint32_t* d_count, const rrt_ray* d_rays, rrt_hit* d_hits,
                             void* stream, std::string* err, int* launches = nullptr) const override;
    int any_hit_indirect(uint64_t capacity, const uint32_t* d_count, const rrt_ray* d_rays, uint8_t* d_occluded,
                         void* stream, std::string* err, int* launches = nullptr) const override;
    const AggregateStats& stats() const override { return stats_; }
    bool literal() const override { return true; }
    // the geometry tables its shape tests read (scene_tables.cuh), which the surface pass reads too
    const ShadeScene& geometry_tables() const;
    void root_bounds(double out6[6]) const {
        for (int k = 0; k < 6; ++k) out6[k] = root_bounds_[k];
    }

  private:
    struct Impl;
    Impl* impl_ = nullptr;
    AggregateStats stats_{};
    double root_bounds_[6] = {0, 0, 0, 0, 0, 0};
    int device_ = 0;
};

}  // namespace rrt

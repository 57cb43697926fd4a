// The device image behind rrt_scene_update_mesh: every primitive of a committed scene baked to world space and kept in
// device memory, so that a mesh update re-bakes only that mesh's primitives on the GPU and the next aggregate is made
// from the image (DeviceAggregate::build_from_image) without the primitives going through the host.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "bvh_lbvh.hpp"
#include "host_scene.hpp"
#include "world_bake.hpp"

namespace rrt {

class MeshImage {
  public:
    MeshImage() = default;
    ~MeshImage();
    MeshImage(const MeshImage&) = delete;
    MeshImage& operator=(const MeshImage&) = delete;

    // Bakes `scene` on the host (bake_world, as a commit does) and uploads the result, with every mesh's positions,
    // vertex indices and primitive runs.
    int create(int device, const HostScene& scene, std::string* err);
    // Mesh `mesh`'s positions on the device, 3 doubles per vertex: an update writes its range there, then calls rebake.
    double* positions(uint32_t mesh) const { return meshes_[mesh].d_p; }
    // Re-bakes every primitive made from mesh `mesh`, bare or under any instance: world vertices, box, fp32-exact flag.
    int rebake(uint32_t mesh, std::string* err);

    // Over all primitives: the world box (the union of the primitive boxes) and whether every vertex is an fp32 value.
    int frame(Aabb* world_box, bool* all_fp32, std::string* err);
    // The Node32 growth sum of DeviceAggregate::build: sum of min(1, cells / half-perimeter) over the primitive boxes.
    int growth(double cells, double* sum, std::string* err);
    // The records in tree order: record `slot` is primitive d_order[slot], as PrimRec48 (wide = false) or PrimRec96,
    // with the fields and the zeroed padding a commit writes.
    int gather(const uint32_t* d_order, bool wide, void* d_records, std::string* err);

    size_t n_prims() const { return n_; }
    const Aabb* boxes() const { return d_box_; }
    LbvhArena& arena() { return arena_; }
    // the tables a DeviceAggregate carries unchanged across mesh updates
    bool has_spheres = false;
    std::vector<double> inst_w2p;
    std::vector<GenSphere> gspheres;

    // primitives [first_prim, first_prim + count) are triangles [first_tri, first_tri + count) of one mesh, under the
    // row-major instance matrix m (has_m) or bare; offset: the run's first thread in a re-bake
    struct Run {
        double m[16];
        uint32_t first_prim, first_tri, count, offset;
        int32_t has_m;
        uint32_t pad;
    };

  private:
    struct Mesh {
        double* d_p = nullptr;
        uint32_t* d_vi = nullptr;
        Run* d_runs = nullptr;
        uint32_t n_runs = 0, n_prims = 0;
    };
    size_t n_ = 0;
    int device_ = 0;
    BakedPrim* d_world_ = nullptr;
    Aabb* d_box_ = nullptr;
    uint8_t* d_kind_ = nullptr;
    uint8_t* d_exact_ = nullptr;
    uint32_t* d_inst_ = nullptr;
    void* d_red_ = nullptr;  // reduction results
    std::vector<Mesh> meshes_;
    LbvhArena arena_;
};

}  // namespace rrt

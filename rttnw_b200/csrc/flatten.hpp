// flatten.hpp — host side: rtx_scene_desc (the reference's object tree as data) ->
// flat device arrays + BVHs. Replaces the pointer-chasing tree walk of
// hittable.rs (List::hit :153-163, BvhTree :260-373) with a layout built for
// coalesced 16-byte loads; the *results* of hit() are the contract, not the
// reference's tree topology (SURVEY.md Q17).
#pragma once
#include <string>
#include <vector>

#include "../../include/rttnw_b200.h"
#include "device_types.h"

namespace rtx {

struct Aabb {
    double lo[3], hi[3];
    void reset();
    void grow(const Aabb& o);
    void grow_point(const double p[3]);
    double half_area() const;
};

struct FlatScene {
    std::vector<BvhNode> nodes;
    std::vector<Record> records;
    std::vector<XformOp> xforms;
    std::vector<DChain> chains;  // chains[0] = identity
    std::vector<DMaterial> materials;
    std::vector<DTexture> textures;
    std::vector<DPerlin> perlins;
    std::vector<DMedium> media;  // in medium-ordinal order
    int32_t max_stack = 0;       // traversal stack entries the deepest root-to-leaf path can need
    // world BVH left to the device builder (lbvh.cuh): records [world_first_record, + world_count) are the world's
    // items in item order, world_boxes holds their fp32 bounds (lo.xyz, hi.xyz; rounded outward), world_root is unset
    bool world_deferred = false;
    int32_t world_first_record = 0, world_count = 0;
    std::vector<float> world_boxes;
    int32_t world_root = 0;
    // the world BVH's nodes are nodes[world_first_node, + world_node_count), root first; world_depth = inner nodes on
    // its longest root-to-leaf path (the shared-memory traversal stages that range and needs one stack entry per level)
    int32_t world_first_node = 0, world_node_count = 0, world_depth = 0;
    int32_t wide_root = -1;      // the same BVH 4-wide (two consecutive BvhNode entries per node), -1: not built
    int32_t n_media = 0;
    int32_t n_prims = 0;  // number of primitive ids handed out
    Aabb world_bounds;
    CameraView camera;
};

// The binned-SAH policy, one definition for the host builder (flatten.cpp) and the device builder (sah_build.cuh).
constexpr int kBvhBins = 16;         // bins per axis (a node of n < 16 primitives gets max(2, n))
constexpr int kBvhMaxLeafLimit = 4;  // largest leaf either builder makes
struct BvhPolicy {
    int max_leaf = 4;            // RTX_BVH_LEAF (1 .. kBvhMaxLeafLimit) overrides, for experiments
    double cost_traverse = 1.0;  // one 64-byte node fetch + two fp32 slab tests
    double cost_prim = 2.0;      // one 96-byte record + an f64 intersection, in units of cost_traverse; RTX_BVH_CPRIM overrides
    static BvhPolicy from_env();
};

// Returns false and fills `err` on malformed input.
// defer_world_bvh: leave the BVH over the world to the device builder when the world has at least two items.
// wide_copy: append the 4-wide copy of the (host-built) world BVH to the node array and set wide_root.
bool flatten_scene(const rtx_scene_desc& desc, FlatScene& out, std::string& err, bool defer_world_bvh = false, bool wide_copy = false);

// Structural invariants of the result (every record inside every ancestor box, every
// record reachable exactly once per BVH, leaf sizes). Host logic test hook.
bool check_flat_scene(const FlatScene& fs, std::string& err);

void camera_view(const rtx_camera& cam, const double background[3], CameraView& out);

}  // namespace rtx

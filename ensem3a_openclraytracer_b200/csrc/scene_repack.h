// Host-side validation and repacking of the reference-layout scene buffers (SURVEY.md §8a) into the layouts
// rt_trace.cuh consumes.  No CUDA calls: b200rt_set_scene uploads the result and commits it to the context only
// after every copy has succeeded.
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

namespace b200rt {

// std::vector that leaves trivially-constructible elements uninitialised on resize(): the repacked arrays of a
// 5 M-triangle scene are ~1 GB, every element is written by the (parallel) loops, and a serial zero-fill first would
// cost more than those loops.
template <class T>
struct raw_alloc : std::allocator<T> {
  template <class U> struct rebind { using other = raw_alloc<U>; };
  raw_alloc() = default;
  template <class U> raw_alloc(const raw_alloc<U> &) {}
  template <class U> void construct(U *p) noexcept { ::new (static_cast<void *>(p)) U; }
  template <class U, class... A> void construct(U *p, A &&...a) { ::new (static_cast<void *>(p)) U(std::forward<A>(a)...); }
};
template <class T> using raw_vector = std::vector<T, raw_alloc<T>>;

// The scalar description of a repacked scene: what the kernels' launch geometry, margins and stacks derive from.  A
// context commits it in one assignment once the scene's buffers are on its GPU.
struct SceneDesc {
  int n_nodes9 = 0, n_inner = 0, n_tris = 0;
  int node_f4 = 2;              // 2 in global memory, 3 when nodes + triangles fit the shared-memory staging area
  int depth = 0, ref_stack_need = 0;   // of the caller's tree
  int cull_depth = 0;           // level of the deepest leaf of the tree `nodes` holds (sizes the traversal stacks)
  bool canonical = true;        // strict two-child tree with nested boxes: the fast traversal applies
  int root_ref = 0;
  float grid_base[3] = {0, 0, 0}, grid_pitch[3] = {1, 1, 1};
  uint32_t root_w[3] = {0x7fff0000u, 0x7fff0000u, 0x7fff0000u};  // the root box as node-record words (max plane << 16 | min plane)
  float cull_abs = 0.0f, cmax = 0.0f;
  int fast_ok = 0;
  float root_box[6] = {0, 0, 0, 0, 0, 0};  // the caller's root box, bvh[2..7] (min.xyz, max.xyz): the denoiser's scale
};

struct Repacked : SceneDesc {
  struct f4 { float x, y, z, w; };
  struct u4 { uint32_t x, y, z, w; };
  raw_vector<u4> nodes;         // node_f4 x 16 bytes per interior node (rt_trace.cuh "repacked scene")
  raw_vector<f4> tris, normals, tboxes;
  raw_vector<f4> ctris;         // the triangle records in the order of the culling tree's leaves (what leaf refs index); .w of the
                                // third vector = the triangle's id
  std::vector<int32_t> tri_mat;
  raw_vector<int32_t> leaf_count;  // per node of the as-is array: leaves in its sub-tree (validate_chain, rt_trace.cuh)
  int cull_tree = 0;            // 0: `nodes` has the caller's topology, 1: the tree of cull_tree.cpp
  double ms_tris = 0, ms_walk = 0, ms_nodes = 0;  // host time of the three stages
};

constexpr size_t kSmemSceneMax = 48 * 1024;  // repacked nodes + triangles up to this size are staged in shared memory
constexpr int kRefStackMax = 64;             // thread-local stack of the exact walk (rt_trace.cuh kRefStack)
constexpr size_t kLaneSmemMax = 96 * 1024;   // room for the per-lane shared-memory stacks of one CTA

// one interior node of a culling tree: the exact boxes (min.xyz, max.xyz) and refs (>= 0 interior index, < 0 ~triangle)
// of its two children
struct CullNode {
  float box[2][6];
  int32_t ref[2];
};

// cull_tree.cpp: binned-SAH tree over the triangles' leaf boxes, nodes in storage order
void build_cull_tree(const Repacked::f4 *tboxes, int n_tris, std::vector<CullNode> *out, int *depth_out);

// bytes of per-lane traversal state in shared memory for a stack of `stack_depth` entries (rt_kernels.cuh lays it out)
size_t lane_smem_bytes_host(int stack_depth);

// Returns 0, or a negative b200rt_status with *err describing the first offending element.
// own_tree: build the culling tree here (cull_tree.cpp) instead of taking the caller's topology over.
int repack_scene(const float *vp, int64_t n_vp, const float *vn, int64_t n_vn, const int32_t *face, int64_t n_face,
                 int64_t n_materials, const float *bvh, int64_t n_bvh, Repacked *out, std::string *err, bool own_tree = true);

}  // namespace b200rt

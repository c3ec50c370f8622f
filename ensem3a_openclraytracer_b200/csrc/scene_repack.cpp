// Validation and repacking of the reference-layout scene (FileManager.py / BVH.py buffers, SURVEY.md §8a) for the
// traversal kernels — host code only, OpenMP over triangles and over interior nodes.  The one serial stage is the
// right-first walk of the tree, which fixes every leaf's rank in the reference's visiting order (MathLib.cl:252-280).
#include "scene_repack.h"

#include <omp.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/b200rt.h"

namespace b200rt {

namespace {

double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

std::string fmt(const char *f, long long a = 0, long long b = 0, long long c = 0) {
  char buf[256];
  snprintf(buf, sizeof buf, f, a, b, c);
  return buf;
}

float as_float(uint32_t u) {
  float f;
  memcpy(&f, &u, 4);
  return f;
}
uint32_t as_u32(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  return u;
}

// The grid of one axis: plane q lies at base + fq * pitch, fq = 0.5 + q / 65536, q in [0, 32767].
struct Axis {
  float base, pitch;
};

double plane_at(const Axis &g, int q) { return (double)g.base + (0.5 + q / 65536.0) * (double)g.pitch; }

// Grid planes (q_min, q_max) that enclose [mn, mx] in real arithmetic, packed as a node-record word.  binary64
// throughout: fq * pitch is exact (16 x 24 bits), the sum with base rounds once (relative 2^-53), and `slack` covers
// that rounding many times over.  Returns false when the grid does not reach that far (a box outside the root box).
bool quantise(const Axis &g, float mn, float mx, uint32_t *w_out) {
  const double base = g.base, pitch = g.pitch;
  const double slack = (std::fabs(base) + pitch) * 0x1p-48;
  double fl = std::floor((((double)mn - base) / pitch - 0.5) * 65536.0);
  double fh = std::ceil((((double)mx - base) / pitch - 0.5) * 65536.0);
  int ql = !(fl >= 0.0) ? 0 : (fl > 32767.0 ? 32767 : (int)fl);
  int qh = !(fh >= 0.0) ? 0 : (fh > 32767.0 ? 32767 : (int)fh);
  while (ql > 0 && plane_at(g, ql) > (double)mn - slack) --ql;
  while (qh < 32767 && plane_at(g, qh) < (double)mx + slack) ++qh;
  *w_out = ((uint32_t)qh << 16) | (uint32_t)ql;
  return plane_at(g, ql) <= (double)mn - slack && plane_at(g, qh) >= (double)mx + slack;
}

}  // namespace

namespace {

// Host threads of the repack.  torchrun exports OMP_NUM_THREADS=1 to every rank "to avoid overload", which would build
// the culling tree of every frame's upload on one core while the rest of the node idles: in that situation — one
// thread allowed and a launcher that says how many ranks share the host — each rank takes its share of the cores
// (at most 16).  B200RT_HOST_THREADS overrides; in every other case OpenMP's own setting stands.
struct HostThreads {
  int saved = 0;
  HostThreads() {
    int want = 0;
    if (const char *q = getenv("B200RT_HOST_THREADS")) {
      want = atoi(q);
    } else if (omp_get_max_threads() == 1) {
      const char *omp = getenv("OMP_NUM_THREADS"), *lws = getenv("LOCAL_WORLD_SIZE");
      if (omp && lws && atoi(omp) == 1 && atoi(lws) >= 1) want = std::min(16, omp_get_num_procs() / atoi(lws));
    }
    if (want >= 1) {
      saved = omp_get_max_threads();
      omp_set_num_threads(want);
    }
  }
  ~HostThreads() {
    if (saved) omp_set_num_threads(saved);
  }
};

}  // namespace

int repack_scene(const float *vp, int64_t n_vp, const float *vn, int64_t n_vn, const int32_t *face, int64_t n_face,
                 int64_t n_materials, const float *bvh, int64_t n_bvh, Repacked *out, std::string *err, bool own_tree) {
  HostThreads host_threads;
  Repacked &R = *out;
  const int n_nodes = (int)(n_bvh / 9), n_tris = (int)(n_face / 10);
  const int nvp = (int)(n_vp / 3), nvn = (int)(n_vn / 3), nm = (int)n_materials;
  R.n_nodes9 = n_nodes;
  R.n_tris = n_tris;
  double t0 = now_ms();

  // ---- triangles: validate indices, precompute edges exactly as MathLib.cl:129-130 rounds them ------------------
  R.tris.resize((size_t)n_tris * 3);
  R.normals.resize((size_t)n_tris);
  R.tboxes.resize((size_t)n_tris * 2);
  R.tri_mat.resize((size_t)n_tris);
  float cmax = 0.0f;
  int first_bad = n_tris;   // first triangle with an out-of-range index
  int nonfinite = 0;
  const float unranked = as_float(0x7fffffffu);
#pragma omp parallel for schedule(static) reduction(max : cmax) reduction(min : first_bad) reduction(| : nonfinite)
  for (int t = 0; t < n_tris; ++t) {
    const int32_t *f = face + 10 * (size_t)t;
    bool ok = f[4] >= 0 && f[4] < nvn && f[0] >= 0 && f[0] < nm;
    for (int j = 7; j < 10; ++j) ok = ok && f[j] >= 0 && f[j] < nvp;
    if (!ok) {
      if (t < first_bad) first_bad = t;
      continue;
    }
    const float *a = vp + 3 * (size_t)f[7], *b = vp + 3 * (size_t)f[8], *c = vp + 3 * (size_t)f[9];
    const float e1x = b[0] - a[0], e1y = b[1] - a[1], e1z = b[2] - a[2];
    const float e2x = c[0] - a[0], e2y = c[1] - a[1], e2z = c[2] - a[2];
    R.tris[3 * (size_t)t + 0] = Repacked::f4{a[0], a[1], a[2], e1x};
    R.tris[3 * (size_t)t + 1] = Repacked::f4{e1y, e1z, e2x, e2y};
    R.tris[3 * (size_t)t + 2] = Repacked::f4{e2z, as_float((uint32_t)f[0]), unranked, 0.0f};
    const float *n0 = vn + 3 * (size_t)f[4];
    R.normals[t] = Repacked::f4{n0[0], n0[1], n0[2], 0.0f};
    R.tboxes[2 * (size_t)t] = Repacked::f4{0, 0, 0, 0};   // stays empty if no leaf holds the triangle
    R.tboxes[2 * (size_t)t + 1] = Repacked::f4{0, 0, 0, 0};
    R.tri_mat[t] = f[0];
    for (int j = 7; j < 10; ++j)
      for (int k = 0; k < 3; ++k) {
        const float v = std::fabs(vp[3 * (size_t)f[j] + k]);
        if (!std::isfinite(v)) nonfinite |= 1;
        else if (v > cmax) cmax = v;
      }
  }
  if (first_bad < n_tris) {
    const int32_t *f = face + 10 * (size_t)first_bad;
    for (int j = 7; j < 10; ++j)
      if (f[j] < 0 || f[j] >= nvp) {
        *err = fmt("triangle %lld: position index %lld out of range [0,%lld)", first_bad, f[j], nvp);
        return B200RT_ERR_INVALID;
      }
    if (f[4] < 0 || f[4] >= nvn) {
      *err = fmt("triangle %lld: normal index %lld out of range [0,%lld)", first_bad, f[4], nvn);
      return B200RT_ERR_INVALID;
    }
    *err = fmt("triangle %lld: material %lld out of range [0,%lld)", first_bad, f[0], nm);
    return B200RT_ERR_INVALID;
  }
  double t1 = now_ms();
  R.ms_tris = t1 - t0;

  // ---- nodes: validate, detect tree shape, rank leaves in the reference's visiting order -----------------------
  std::vector<int> inner_id((size_t)n_nodes, -1);
  std::vector<unsigned char> seen((size_t)n_nodes, 0);
  bool canonical = true;
  auto L = [&](int i) { return (int)bvh[9 * (size_t)i]; };
  auto Rc = [&](int i) { return (int)bvh[9 * (size_t)i + 1]; };
  auto T = [&](int i) { return (int)bvh[9 * (size_t)i + 8]; };
  int depth = 0;
  size_t max_stack = 1;
  std::vector<int> first_rank;    // id-ordered trees: rank of the first leaf under each node
  // ---- fast path: a tree whose children always carry larger ids than their parent (what BVH.py and the native
  // builder emit: children are appended at split time).  Everything the serial walk below derives then follows from
  // passes over the node array in id order — per-node checks in parallel, depth / pending-stack / first-rank top-down,
  // leaves per sub-tree bottom-up — instead of one pointer-chasing walk over ten million nodes.
  bool id_ordered = n_nodes >= 1;
  {
    int bad = 0, noncanon = 0, nf = 0;
    float cm = cmax;
    std::vector<int> indeg((size_t)n_nodes, 0);
#pragma omp parallel for schedule(static) reduction(| : bad, noncanon, nf) reduction(max : cm)
    for (int i = 0; i < n_nodes; ++i) {
      const float *rec = bvh + 9 * (size_t)i;
      const int l = (int)rec[0], r = (int)rec[1], t = (int)rec[8];
      if (t < -1 || t >= n_tris || l < -1 || r < -1 || l >= n_nodes || r >= n_nodes || (l != -1 && l <= i) || (r != -1 && r <= i) ||
          (l != -1 && l == r)) {
        bad |= 1;
        continue;
      }
      const float *bx = rec + 2;
      for (int k = 0; k < 6; ++k) {
        const float v = std::fabs(bx[k]);
        if (!std::isfinite(v)) nf |= 1;
        else if (v > cm) cm = v;
      }
      const bool leaf = (t != -1 && l == -1 && r == -1), inner = (t == -1 && l != -1 && r != -1);
      if (!leaf && !inner) noncanon |= 1;
      for (int k = 0; k < 3; ++k)
        if (!(bx[k] <= bx[k + 3])) noncanon |= 1;
      for (int ch : {l, r})
        if (ch != -1) {
          const float *cb = bvh + 9 * (size_t)ch + 2;
          for (int k = 0; k < 3; ++k)
            if (!(cb[k] >= bx[k] && cb[k + 3] <= bx[k + 3])) noncanon |= 1;
#pragma omp atomic
          indeg[ch]++;
        }
    }
    if (bad) id_ordered = false;
    if (id_ordered) {
      int wrong = indeg[0] != 0 ? 1 : 0;
#pragma omp parallel for schedule(static) reduction(| : wrong)
      for (int i = 1; i < n_nodes; ++i)
        if (indeg[i] != 1) wrong |= 1;   // unreachable or shared nodes: let the walk below decide what to report
      if (wrong) id_ordered = false;
    }
    if (id_ordered) {
      if (nf) nonfinite |= 1;
      if (noncanon) canonical = false;
      cmax = cm;
      // top-down in id order: level, entries pending on the reference's stack when the node is popped, first leaf rank
      std::vector<int> level((size_t)n_nodes, 0), pending((size_t)n_nodes, 0);
      R.leaf_count.resize((size_t)n_nodes);
      for (int i = n_nodes - 1; i >= 0; --i) {
        const float *rec = bvh + 9 * (size_t)i;
        const int l = (int)rec[0], r = (int)rec[1];
        R.leaf_count[i] = ((int)rec[8] != -1 ? 1 : 0) + (l != -1 ? R.leaf_count[l] : 0) + (r != -1 ? R.leaf_count[r] : 0);
      }
      first_rank.assign((size_t)n_nodes, 0);
      for (int i = 0; i < n_nodes; ++i) {
        const float *rec = bvh + 9 * (size_t)i;
        const int l = (int)rec[0], r = (int)rec[1];
        if (level[i] > depth) depth = level[i];
        const size_t pushed = (size_t)pending[i] + (l != -1 ? 1 : 0) + (r != -1 ? 1 : 0);
        if (pushed > max_stack) max_stack = pushed;
        // the reference pushes left then right and pops right first (MathLib.cl:275-280): the right sub-tree is walked
        // with the left child still on the stack and takes the lower ranks; a node's own triangle comes before both
        const int own = (int)rec[8] != -1 ? 1 : 0;
        if (r != -1) {
          level[r] = level[i] + 1;
          pending[r] = pending[i] + (l != -1 ? 1 : 0);
          first_rank[r] = first_rank[i] + own;
        }
        if (l != -1) {
          level[l] = level[i] + 1;
          pending[l] = pending[i];
          first_rank[l] = first_rank[i] + own + (r != -1 ? R.leaf_count[r] : 0);
        }
      }
      int dup = 0;
#pragma omp parallel for schedule(static) reduction(| : dup)
      for (int i = 0; i < n_nodes; ++i) {
        const float *rec = bvh + 9 * (size_t)i;
        const int t = (int)rec[8];
        if (t == -1) continue;
        uint32_t *slot = reinterpret_cast<uint32_t *>(&R.tris[3 * (size_t)t + 2].z);
        uint32_t old;
#pragma omp atomic capture
        { old = *slot; *slot = (uint32_t)first_rank[i]; }
        if (old != 0x7fffffffu) { dup |= 1; continue; }   // a triangle held by two leaves: rank and box ambiguous
        R.tboxes[2 * (size_t)t] = Repacked::f4{rec[2], rec[3], rec[4], 0.0f};
        R.tboxes[2 * (size_t)t + 1] = Repacked::f4{rec[5], rec[6], rec[7], 0.0f};
      }
      if (dup) canonical = false;
    }
  }
  std::vector<int> preorder;
  if (!id_ordered) {
  preorder.reserve((size_t)n_nodes);
  {
    // right-first pre-order walk == the order MathLib.cl:252-280 pops nodes when every box test passes
    struct Item { int node, level; };
    std::vector<Item> stack;
    stack.push_back({0, 0});
    int rank = 0;
    while (!stack.empty()) {
      const Item it = stack.back();
      stack.pop_back();
      const int cur = it.node;
      if (cur < 0 || cur >= n_nodes) {
        *err = fmt("BVH child index %lld out of range [0,%lld)", cur, n_nodes);
        return B200RT_ERR_INVALID;
      }
      if (seen[cur]) {
        *err = fmt("BVH node %lld is reachable twice: not a tree (the traversal would not terminate)", cur);
        return B200RT_ERR_INVALID;
      }
      seen[cur] = 1;
      preorder.push_back(cur);
      const float *rec = bvh + 9 * (size_t)cur;
      const int l = (int)rec[0], r = (int)rec[1], t = (int)rec[8];
      if (t < -1 || t >= n_tris) {
        *err = fmt("BVH node %lld: triangle %lld out of range [0,%lld)", cur, t, n_tris);
        return B200RT_ERR_INVALID;
      }
      if (l < -1 || r < -1) {
        *err = fmt("BVH node %lld: negative child index", cur);
        return B200RT_ERR_INVALID;
      }
      const float *bx = rec + 2;
      for (int k = 0; k < 6; ++k) {
        const float v = std::fabs(bx[k]);
        if (!std::isfinite(v)) nonfinite |= 1;
        else if (v > cmax) cmax = v;
      }
      const bool leaf = (t != -1 && l == -1 && r == -1), inner = (t == -1 && l != -1 && r != -1);
      if (!leaf && !inner) canonical = false;
      // the fast traversal's "leaf passes => ancestors pass" argument needs min <= max and child boxes nested in
      // their parent's (rt_trace.cuh); BVH.py guarantees both, anything else is walked in reference order
      for (int k = 0; k < 3; ++k)
        if (!(bx[k] <= bx[k + 3])) canonical = false;
      for (int ch : {l, r})
        if (ch >= 0 && ch < n_nodes) {
          const float *cb = bvh + 9 * (size_t)ch + 2;
          for (int k = 0; k < 3; ++k)
            if (!(cb[k] >= bx[k] && cb[k + 3] <= bx[k + 3])) canonical = false;
        }
      if (t != -1) {
        Repacked::f4 &t2 = R.tris[3 * (size_t)t + 2];
        if (as_u32(t2.z) == 0x7fffffffu) {
          t2.z = as_float((uint32_t)rank);
          R.tboxes[2 * (size_t)t] = Repacked::f4{bx[0], bx[1], bx[2], 0.0f};
          R.tboxes[2 * (size_t)t + 1] = Repacked::f4{bx[3], bx[4], bx[5], 0.0f};
        } else {
          canonical = false;  // a triangle held by two leaves: rank and leaf box would be ambiguous
        }
        ++rank;
      }
      if (it.level > depth) depth = it.level;
      if (l != -1) stack.push_back({l, it.level + 1});
      if (r != -1) stack.push_back({r, it.level + 1});
      if (stack.size() > max_stack) max_stack = stack.size();
    }
  }
  // leaves per sub-tree: children come after their parent in the pre-order, so the reverse order is bottom-up
  R.leaf_count.assign((size_t)n_nodes, 0);
  for (size_t q = preorder.size(); q-- > 0;) {
    const int cur = preorder[q];
    const float *rec = bvh + 9 * (size_t)cur;
    const int l = (int)rec[0], r = (int)rec[1];
    R.leaf_count[cur] = ((int)rec[8] != -1 ? 1 : 0) + (l != -1 ? R.leaf_count[l] : 0) + (r != -1 ? R.leaf_count[r] : 0);
  }
  }  // !id_ordered
  if (nonfinite) {
    *err = "scene contains a non-finite coordinate (vertex or box plane)";
    return B200RT_ERR_INVALID;
  }
  R.depth = depth;
  R.cull_depth = depth;
  R.cull_tree = 0;
  R.ref_stack_need = (int)max_stack;
  if (R.ref_stack_need > kRefStackMax) canonical = false;  // closest_hit_nodrop's thread-local stack
  double t2 = now_ms();
  R.ms_walk = t2 - t1;

  // ---- the culling tree: built here over the leaf boxes (cull_tree.cpp), or the caller's topology ------------------
  std::vector<CullNode> cull;
  if (canonical && own_tree && T(0) == -1) {
    build_cull_tree(R.tboxes.data(), n_tris, &cull, &R.cull_depth);
    R.cull_tree = 1;
  }
  // a pathologically deep tree would not leave room for the per-lane stacks in shared memory
  if (lane_smem_bytes_host(R.cull_depth + 2) > kLaneSmemMax) canonical = false;

  // ---- grid of the quantised node boxes ------------------------------------------------------------------
  Axis grid[3];
  {
    double ext[3], ext_max = 0.0;
    for (int k = 0; k < 3; ++k) {
      ext[k] = std::max(0.0, (double)bvh[5 + k] - (double)bvh[2 + k]);
      ext_max = std::max(ext_max, ext[k]);
    }
    if (ext_max == 0.0) ext_max = std::max((double)cmax, 1e-30) * 0x1p-12;
    for (int k = 0; k < 3; ++k) {
      const double e = std::max(ext[k], ext_max / 256.0);   // bounded anisotropy: a flat scene keeps a usable pitch
      // plane 0 just below the root's min, plane 32767 just above its max; the span is widened until both hold with the
      // float32 roundings of base and pitch (a scene far from the origin relative to its size needs several ulps)
      double widen = 0x1p-20;
      for (int attempt = 0;; ++attempt) {
        float pitch = (float)(e * (65536.0 / 32767.0) * (1.0 + 8.0 * widen));
        if (!(pitch > 0.0f) || !std::isfinite(pitch)) pitch = 1.0f;
        float base = (float)((double)bvh[2 + k] - 2.0 * widen * e - 0.5 * (double)pitch);
        base = std::nextafterf(base, -INFINITY);
        if (!std::isfinite(base)) base = 0.0f;
        grid[k] = Axis{base, pitch};
        if (quantise(grid[k], bvh[2 + k], bvh[5 + k], &R.root_w[k]) || attempt == 24) break;
        widen *= 4.0;
      }
      R.grid_base[k] = grid[k].base;
      R.grid_pitch[k] = grid[k].pitch;
      const float hi = std::fabs(grid[k].base + grid[k].pitch) * (1.0f + 0x1p-20f), lo = std::fabs(grid[k].base);
      cmax = std::max(cmax, std::max(hi, lo));
    }
    const float dx = bvh[5] - bvh[2], dy = bvh[6] - bvh[3], dz = bvh[7] - bvh[4];
    R.cull_abs = 1e-3f * std::sqrt(dx * dx + dy * dy + dz * dz);
    for (int k = 0; k < 6; ++k) R.root_box[k] = bvh[2 + k];
  }
  R.cmax = cmax;
  // range the conservative slab test's error margin is proven for (rt_trace.cuh); outside it every ray takes
  // closest_hit_nodrop
  R.fast_ok = (cmax <= 1.099511627776e12f /* 2^40 */ && cmax >= 9.5367431640625e-07f /* 2^-20 */) ? 1 : 0;

  // ---- repack interior nodes into the 32-byte two-child records ---------------------------------------------------
  // Order: a node's interior children are adjacent, and a pair is followed by the sub-tree of its first member
  // (pre-order over sibling pairs), so that the 128-byte line that holds a node usually holds the next node of a
  // descent as well — what matters once the tree no longer fits the caches (BASELINE config 5).
  R.nodes.clear();
  R.n_inner = 0;
  R.root_ref = 0;
  R.canonical = canonical;
  if (canonical) {
    if (T(0) != -1) {
      R.root_ref = ~T(0);
    } else {
      std::vector<int> order;
      if (!R.cull_tree) {
      order.reserve((size_t)n_nodes / 2 + 1);
      order.push_back(0);
      inner_id[0] = 0;
      if (id_ordered) {
        // BVH.py appends both children at split time and then builds the left sub-tree completely (BVH.py:107-109,
        // 147-153): interior nodes in id order ARE the pre-order over sibling pairs
        order.clear();
        for (int i = 0; i < n_nodes; ++i)
          if (T(i) == -1) {
            inner_id[i] = (int)order.size();
            order.push_back(i);
          }
      } else {
        std::vector<int> todo;
        todo.push_back(0);
        while (!todo.empty()) {
          const int cur = todo.back();
          todo.pop_back();
          const int ch[2] = {L(cur), Rc(cur)};
          for (int k = 0; k < 2; ++k)
            if (T(ch[k]) == -1) {
              inner_id[ch[k]] = (int)order.size();
              order.push_back(ch[k]);
            }
          for (int k = 1; k >= 0; --k)
            if (T(ch[k]) == -1) todo.push_back(ch[k]);
        }
      }
      }
      // Leaf refs index `ctris`: the triangle records once more, in the order the leaves appear in the node records, so
      // that the leaves of a sub-tree — the triangles neighbouring rays test — share cache lines whatever the order of
      // the caller's face list.
      std::vector<int> leaf_pos;
      if (R.cull_tree) {
        leaf_pos.assign((size_t)n_tris, -1);
        int pos = 0;
        for (size_t q = 0; q < cull.size(); ++q)
          for (int k = 0; k < 2; ++k)
            if (cull[q].ref[k] < 0) leaf_pos[(size_t)~cull[q].ref[k]] = pos++;
      }
      const int n_inner = R.cull_tree ? (int)cull.size() : (int)order.size();
      R.n_inner = n_inner;
      // small scenes are staged in shared memory with 48-byte node spacing (SceneView::node_f4)
      const int nf4 = ((size_t)n_inner * 48 + (size_t)n_tris * 48 <= kSmemSceneMax) ? 3 : 2;
      R.node_f4 = nf4;
      R.nodes.resize((size_t)n_inner * nf4);
      int outside = 0;   // a box the grid over the root box cannot enclose
#pragma omp parallel for schedule(static) reduction(| : outside)
      for (int q = 0; q < n_inner; ++q) {
        const float *bl, *br;   // min.xyz, max.xyz of the two children
        int32_t refl, refr;     // interior refs are 16-byte offsets into the node array (index x 16-byte units per node)
        if (R.cull_tree) {
          const CullNode &N = cull[q];
          bl = N.box[0]; br = N.box[1];
          refl = N.ref[0] < 0 ? ~leaf_pos[(size_t)~N.ref[0]] : N.ref[0] * nf4;
          refr = N.ref[1] < 0 ? ~leaf_pos[(size_t)~N.ref[1]] : N.ref[1] * nf4;
        } else {
          const int cur = order[q];
          const int l = L(cur), r = Rc(cur);
          bl = bvh + 9 * (size_t)l + 2; br = bvh + 9 * (size_t)r + 2;
          refl = T(l) != -1 ? ~T(l) : (int32_t)(inner_id[l] * nf4);
          refr = T(r) != -1 ? ~T(r) : (int32_t)(inner_id[r] * nf4);
        }
        uint32_t wl[3], wr[3];
        for (int k = 0; k < 3; ++k)
          if (!quantise(grid[k], bl[k], bl[3 + k], &wl[k]) || !quantise(grid[k], br[k], br[3 + k], &wr[k])) outside |= 1;
        Repacked::u4 a, b;
        a.x = wl[0]; a.y = wl[1]; a.z = wl[2]; a.w = wr[0];
        b.x = wr[1]; b.y = wr[2];
        b.z = (uint32_t)refl;
        b.w = (uint32_t)refr;
        R.nodes[(size_t)nf4 * q + 0] = a;
        R.nodes[(size_t)nf4 * q + 1] = b;
        if (nf4 == 3) R.nodes[(size_t)nf4 * q + 2] = Repacked::u4{0, 0, 0, 0};
      }
      if (R.cull_tree) {
        R.ctris.resize((size_t)n_tris * 3);
#pragma omp parallel for schedule(static)
        for (int t = 0; t < n_tris; ++t) {
          const size_t p = (size_t)leaf_pos[(size_t)t];
          R.ctris[3 * p] = R.tris[3 * (size_t)t];
          R.ctris[3 * p + 1] = R.tris[3 * (size_t)t + 1];
          Repacked::f4 t2 = R.tris[3 * (size_t)t + 2];
          t2.w = as_float((uint32_t)t);
          R.ctris[3 * p + 2] = t2;
        }
      }
      if (outside) {   // cannot happen for nested boxes; such a tree is walked in reference order
        R.canonical = false;
        R.nodes.clear();
        R.n_inner = 0;
        R.node_f4 = 2;
      }
    }
  }
  if (R.ctris.size() != R.tris.size() || !R.cull_tree || !R.canonical) {   // leaf refs are triangle ids
    R.ctris.resize(R.tris.size());
#pragma omp parallel for schedule(static)
    for (int t = 0; t < n_tris; ++t) {
      R.ctris[3 * (size_t)t] = R.tris[3 * (size_t)t];
      R.ctris[3 * (size_t)t + 1] = R.tris[3 * (size_t)t + 1];
      Repacked::f4 t2 = R.tris[3 * (size_t)t + 2];
      t2.w = as_float((uint32_t)t);
      R.ctris[3 * (size_t)t + 2] = t2;
    }
  }
  R.ms_nodes = now_ms() - t2;
  return 0;
}

}  // namespace b200rt

extern "C" int b200rt_repack_probe(const float *vp, int64_t n_vp, const float *vn, int64_t n_vn, const int32_t *face,
                                   int64_t n_face, int64_t n_materials, const float *bvh, int64_t n_bvh,
                                   uint32_t *nodes_out, int64_t n_nodes_out, int32_t *rank_out, float *info) {
  if (!vp || !vn || !face || !bvh || !info || n_vp <= 0 || n_vp % 3 || n_vn <= 0 || n_vn % 3 || n_face <= 0 || n_face % 10 ||
      n_bvh <= 0 || n_bvh % 9 || n_materials <= 0)
    return B200RT_ERR_INVALID;
  b200rt::Repacked R;
  std::string msg;
  const char *own = getenv("B200RT_CULL_TREE");
  int rc = b200rt::repack_scene(vp, n_vp, vn, n_vn, face, n_face, n_materials, bvh, n_bvh, &R, &msg, !(own && own[0] == '0'));
  if (rc) return rc;
  info[0] = (float)R.n_inner; info[1] = (float)R.node_f4; info[2] = (float)R.depth; info[3] = (float)R.ref_stack_need;
  info[4] = R.canonical ? 1.0f : 0.0f; info[5] = (float)R.fast_ok; info[6] = R.cmax; info[7] = R.cull_abs;
  for (int k = 0; k < 3; ++k) {
    info[8 + k] = R.grid_base[k]; info[11 + k] = R.grid_pitch[k];
    info[14 + k] = (float)(R.root_w[k] & 0xffffu); info[17 + k] = (float)(R.root_w[k] >> 16);   // root box: min / max plane index
  }
  info[20] = (float)R.ms_tris; info[21] = (float)R.ms_walk; info[22] = (float)R.ms_nodes; info[23] = (float)R.cull_depth;
  if (rank_out)
    for (int t = 0; t < R.n_tris; ++t) memcpy(&rank_out[t], &R.tris[3 * (size_t)t + 2].z, 4);
  if (nodes_out) {
    if (n_nodes_out < (int64_t)R.n_inner * 8) return B200RT_ERR_INVALID;
    for (int q = 0; q < R.n_inner; ++q) {
      const b200rt::Repacked::u4 &a = R.nodes[(size_t)R.node_f4 * q], &b = R.nodes[(size_t)R.node_f4 * q + 1];
      uint32_t *o = nodes_out + 8 * (size_t)q;
      o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
      for (int k = 6; k < 8; ++k)   // leaf refs index `ctris`: reported as the triangle they stand for
        if ((int32_t)o[k] < 0) {
          uint32_t id;
          memcpy(&id, &R.ctris[3 * (size_t)~(int32_t)o[k] + 2].w, 4);
          o[k] = (uint32_t)~(int32_t)id;
        }
    }
  }
  return 0;
}

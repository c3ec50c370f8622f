// The culling tree of the fast traversal: a binary tree over the LEAF BOXES of the caller's BVH, built here with a
// binned surface-area heuristic instead of taken over from the caller's array.
//
// Why this is allowed.  The reference accepts a triangle iff the exact slab test passes for its leaf box and every
// ancestor box of ITS tree and Möller–Trumbore accepts it (MathLib.cl:234-288); for the rays the fast traversal walks,
// the leaf box decides (rt_trace.cuh, top).  The interior boxes therefore only cull, and any tree whose boxes are unions
// of the reference's leaf boxes culls correctly: a box that encloses a leaf box cannot fail the conservative test when
// the leaf box passes the exact one.  Which triangle wins a tie, the exact test of the winner's leaf box, the chain
// validation of irregular rays and the exact re-trace all keep using the caller's tree (ranks, `tboxes`, `bvh9`).
//
// Why it pays.  BVH.py splits every node at the mean centroid along the axis of largest variance (BVH.py:75-109); on
// scenes with long thin triangles (Serre_leger) that leaves sibling boxes overlapping almost completely.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>

#include "scene_repack.h"

namespace b200rt {

namespace {

constexpr int kBins = 32;             // SAH bins per axis
constexpr int kSahLevels = 64;        // below this level ranges are halved by index: bounds the depth at 64 + log2(n)
constexpr int kTaskMin = 256;         // sub-trees smaller than this are built by the task that reached them
constexpr int kParallelBin = 1 << 18; // ranges larger than this are binned by several tasks

struct Box {
  float mn[3], mx[3];
  void reset() {
    for (int k = 0; k < 3; ++k) { mn[k] = INFINITY; mx[k] = -INFINITY; }
  }
  void grow(const float *lo, const float *hi) {
    for (int k = 0; k < 3; ++k) {
      mn[k] = std::min(mn[k], lo[k]);
      mx[k] = std::max(mx[k], hi[k]);
    }
  }
  void grow(const Box &b) { grow(b.mn, b.mx); }
  double half_area() const {
    const double dx = (double)mx[0] - mn[0], dy = (double)mx[1] - mn[1], dz = (double)mx[2] - mn[2];
    return dx * dy + dy * dz + dz * dx;
  }
};

struct Bins {
  Box box[3][kBins];
  int cnt[3][kBins];
  void reset(int nb) {
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < nb; ++b) { box[a][b].reset(); cnt[a][b] = 0; }
  }
  void merge(const Bins &o, int nb) {
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < nb; ++b)
        if (o.cnt[a][b]) { box[a][b].grow(o.box[a][b]); cnt[a][b] += o.cnt[a][b]; }
  }
};

// The builder partitions the leaf boxes themselves, not indices into them: every pass over a range is then a sequential
// sweep (with an index array the upper levels of a 5 M-triangle tree gather 160 MB at random, level after level).
struct Prim {
  float mn[3], mx[3];
  int32_t id;
  int32_t pad;
};

struct Builder {
  Prim *prim;
  CullNode *nodes;
  std::atomic<int> next{0};
  std::atomic<int> depth{0};

  static float centre(const Prim &p, int a) { return 0.5f * p.mn[a] + 0.5f * p.mx[a]; }

  static int bin_of(float c, float c0, float scale, int nb) {
    int b = (int)((c - c0) * scale);
    return b < 0 ? 0 : (b >= nb ? nb - 1 : b);
  }

  void bin_range(int begin, int end, const float *c0, const float *scale, int nb, Bins *out) const {
    out->reset(nb);
    for (int i = begin; i < end; ++i) {
      const Prim &p = prim[i];
      for (int a = 0; a < 3; ++a) {
        if (!(scale[a] > 0.0f)) continue;
        const int b = bin_of(centre(p, a), c0[a], scale[a], nb);
        out->box[a][b].grow(p.mn, p.mx);
        out->cnt[a][b]++;
      }
    }
  }

  // builds the sub-tree over prim[begin, end) (end - begin >= 2); returns its interior index and box
  int build(int begin, int end, int level, Box *box_out) {
    const int n = end - begin;
    const int me = next.fetch_add(1, std::memory_order_relaxed);
    CullNode &N = nodes[me];
    int mid = begin + n / 2;
    if (n > 2 && level < kSahLevels) {
      // centroid bounds
      float c0[3] = {INFINITY, INFINITY, INFINITY}, c1[3] = {-INFINITY, -INFINITY, -INFINITY};
      for (int i = begin; i < end; ++i)
        for (int a = 0; a < 3; ++a) {
          const float c = centre(prim[i], a);
          c0[a] = std::min(c0[a], c);
          c1[a] = std::max(c1[a], c);
        }
      // a range of a few triangles does not need (and should not pay for clearing and sweeping) all the bins
      const int nb = std::min(kBins, std::max(4, 2 * n));
      float scale[3];
      bool any = false;
      for (int a = 0; a < 3; ++a) {
        const float e = c1[a] - c0[a];
        scale[a] = (e > 0.0f && std::isfinite(e)) ? (float)nb * (1.0f - 0x1p-20f) / e : 0.0f;
        if (!std::isfinite(scale[a])) scale[a] = 0.0f;
        any = any || scale[a] > 0.0f;
      }
      if (any) {
        Bins B;
        if (n >= kParallelBin) {
          constexpr int kParts = 16;
          std::vector<Bins> part(kParts);
          for (int p = 0; p < kParts; ++p) {
            const int b0 = begin + (int)((long long)n * p / kParts), b1 = begin + (int)((long long)n * (p + 1) / kParts);
            Bins *dst = &part[p];
#pragma omp task firstprivate(b0, b1, dst, nb) shared(c0, scale)
            bin_range(b0, b1, c0, scale, nb, dst);
          }
#pragma omp taskwait
          B.reset(nb);
          for (int p = 0; p < kParts; ++p) B.merge(part[p], nb);
        } else {
          bin_range(begin, end, c0, scale, nb, &B);
        }
        double best = INFINITY;
        int best_axis = -1, best_split = 0;
        for (int a = 0; a < 3; ++a) {
          if (!(scale[a] > 0.0f)) continue;
          double right_area[kBins];
          int right_cnt[kBins];
          Box acc;
          acc.reset();
          int c = 0;
          for (int b = nb - 1; b > 0; --b) {
            if (B.cnt[a][b]) acc.grow(B.box[a][b]);
            c += B.cnt[a][b];
            right_area[b] = c ? acc.half_area() : 0.0;
            right_cnt[b] = c;
          }
          acc.reset();
          c = 0;
          for (int b = 0; b < nb - 1; ++b) {   // split after bin b
            if (B.cnt[a][b]) acc.grow(B.box[a][b]);
            c += B.cnt[a][b];
            if (c == 0 || right_cnt[b + 1] == 0) continue;
            const double cost = acc.half_area() * c + right_area[b + 1] * right_cnt[b + 1];
            if (cost < best) { best = cost; best_axis = a; best_split = b; }
          }
        }
        if (best_axis >= 0) {
          const int a = best_axis;
          const float a0 = c0[a], sc = scale[a];
          Prim *m = std::partition(prim + begin, prim + end, [&](const Prim &q) { return bin_of(centre(q, a), a0, sc, nb) <= best_split; });
          mid = (int)(m - prim);
          if (mid == begin || mid == end) mid = begin + n / 2;   // cannot happen (both sides counted); keep the build total
        }
      }
    }
    Box bl, br;
    int refl, refr;
    const bool spawn = n >= kTaskMin;
    if (mid - begin == 1) {
      refl = ~prim[begin].id;
      bl.reset(); bl.grow(prim[begin].mn, prim[begin].mx);
      if (level + 1 > depth.load(std::memory_order_relaxed)) bump_depth(level + 1);
    } else if (spawn) {
#pragma omp task shared(refl, bl) firstprivate(begin, mid, level)
      refl = build(begin, mid, level + 1, &bl);
    } else {
      refl = build(begin, mid, level + 1, &bl);
    }
    if (end - mid == 1) {
      refr = ~prim[mid].id;
      br.reset(); br.grow(prim[mid].mn, prim[mid].mx);
      if (level + 1 > depth.load(std::memory_order_relaxed)) bump_depth(level + 1);
    } else {
      refr = build(mid, end, level + 1, &br);
    }
    if (spawn) {
#pragma omp taskwait
    }
    N.ref[0] = refl;
    N.ref[1] = refr;
    for (int k = 0; k < 3; ++k) {
      N.box[0][k] = bl.mn[k]; N.box[0][3 + k] = bl.mx[k];
      N.box[1][k] = br.mn[k]; N.box[1][3 + k] = br.mx[k];
    }
    box_out->reset();
    box_out->grow(bl);
    box_out->grow(br);
    return me;
  }

  void bump_depth(int d) {
    int cur = depth.load(std::memory_order_relaxed);
    while (d > cur && !depth.compare_exchange_weak(cur, d, std::memory_order_relaxed)) {}
  }
};

}  // namespace

// tboxes: the leaf box of every triangle (2 x f4: min, max).  out: n_tris - 1 interior nodes, node 0 the root, a node's
// interior children adjacent and a pair followed by the sub-tree of its first member (the order the node records are
// stored in: the 128-byte line that holds a node usually holds the next node of a descent as well).  *depth_out: level
// of the deepest leaf (root = level 0), which bounds the entries the near-first walk keeps on its stack.
void build_cull_tree(const Repacked::f4 *tboxes, int n_tris, std::vector<CullNode> *out, int *depth_out) {
  out->clear();
  *depth_out = 0;
  if (n_tris < 2) return;
  std::vector<Prim> prim((size_t)n_tris);
#pragma omp parallel for schedule(static)
  for (int i = 0; i < n_tris; ++i) {
    const Repacked::f4 &lo = tboxes[2 * (size_t)i], &hi = tboxes[2 * (size_t)i + 1];
    prim[i] = Prim{{lo.x, lo.y, lo.z}, {hi.x, hi.y, hi.z}, i, 0};
  }
  std::vector<CullNode> tmp((size_t)n_tris - 1);
  Builder B;
  B.prim = prim.data();
  B.nodes = tmp.data();
  Box root;
#pragma omp parallel
#pragma omp single
  B.build(0, n_tris, 0, &root);
  *depth_out = B.depth.load();
  const int n_inner = n_tris - 1;

  // ---- tree rotations: a child changes places with a grandchild on the other side where that shrinks the box in between
  // (bottom-up sweeps until nothing improves; the root's box and every leaf box stay what they were)
  const int passes = n_tris > 1000000 ? 1 : 2;   // the sweeps are serial: one is most of the gain
  {
    auto area6 = [](const float *b) {
      const double dx = (double)b[3] - b[0], dy = (double)b[4] - b[1], dz = (double)b[5] - b[2];
      return dx * dy + dy * dz + dz * dx;
    };
    std::vector<int> post;
    post.reserve((size_t)n_inner);
    {
      std::vector<int> st;
      st.push_back(0);
      while (!st.empty()) {     // reverse pre-order = children before parents
        const int cur = st.back();
        st.pop_back();
        post.push_back(cur);
        for (int k = 0; k < 2; ++k)
          if (tmp[cur].ref[k] >= 0) st.push_back(tmp[cur].ref[k]);
      }
    }
    for (int pass = 0; pass < passes; ++pass) {
      long long changed = 0;
      for (size_t q = post.size(); q-- > 0;) {
        CullNode &N = tmp[post[q]];
        double best_gain = 0.0;
        int best_s = -1, best_g = -1;
        float best_box[6];
        for (int s = 0; s < 2; ++s) {
          if (N.ref[s] < 0) continue;
          const CullNode &X = tmp[N.ref[s]];
          const float *y = N.box[1 - s];
          const double ax = area6(N.box[s]);
          for (int g = 0; g < 2; ++g) {       // the other side's child changes places with X's child g
            const float *keep = X.box[1 - g];
            float u[6];
            for (int k = 0; k < 3; ++k) { u[k] = std::min(y[k], keep[k]); u[3 + k] = std::max(y[3 + k], keep[3 + k]); }
            const double gain = ax - area6(u);
            if (gain > best_gain) { best_gain = gain; best_s = s; best_g = g; memcpy(best_box, u, sizeof u); }
          }
        }
        if (best_s < 0) continue;
        CullNode &X = tmp[N.ref[best_s]];
        const int y_ref = N.ref[1 - best_s];
        float y_box[6];
        memcpy(y_box, N.box[1 - best_s], sizeof y_box);
        N.ref[1 - best_s] = X.ref[best_g];
        memcpy(N.box[1 - best_s], X.box[best_g], sizeof y_box);
        X.ref[best_g] = y_ref;
        memcpy(X.box[best_g], y_box, sizeof y_box);
        memcpy(N.box[best_s], best_box, sizeof best_box);
        ++changed;
      }
      if (!changed) break;
    }
    // levels moved: the depth again
    std::vector<std::pair<int, int>> st;
    st.push_back({0, 0});
    int deepest = 0;
    while (!st.empty()) {
      const auto cur = st.back();
      st.pop_back();
      for (int k = 0; k < 2; ++k) {
        if (tmp[cur.first].ref[k] >= 0) st.push_back({tmp[cur.first].ref[k], cur.second + 1});
        else deepest = std::max(deepest, cur.second + 1);
      }
    }
    *depth_out = deepest;
  }

  // final order: pre-order over sibling pairs
  std::vector<int> pos((size_t)n_inner, -1), order;
  order.reserve((size_t)n_inner);
  order.push_back(0);
  pos[0] = 0;
  std::vector<int> todo;
  todo.push_back(0);
  while (!todo.empty()) {
    const int cur = todo.back();
    todo.pop_back();
    const CullNode &N = tmp[cur];
    for (int k = 0; k < 2; ++k)
      if (N.ref[k] >= 0) {
        pos[N.ref[k]] = (int)order.size();
        order.push_back(N.ref[k]);
      }
    for (int k = 1; k >= 0; --k)
      if (N.ref[k] >= 0) todo.push_back(N.ref[k]);
  }
  out->resize((size_t)n_inner);
#pragma omp parallel for schedule(static)
  for (int q = 0; q < n_inner; ++q) {
    CullNode N = tmp[order[q]];
    for (int k = 0; k < 2; ++k)
      if (N.ref[k] >= 0) N.ref[k] = pos[N.ref[k]];
    (*out)[q] = N;
  }
}

}  // namespace b200rt

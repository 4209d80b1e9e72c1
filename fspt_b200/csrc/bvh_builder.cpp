// bvh_builder.cpp -- native, multi-threaded builder that reproduces the reference's JavaScript BVH
// (bvh.js:5-198) and its pre-order flatten (bvh.js:33-50, main.js:366-392) bit for bit.
//
// Same tree, different machinery: instead of one JS object per node holding three freshly sliced index
// lists and a Set per split, the three centroid-sorted index arrays are partitioned IN PLACE (stable),
// every node owns a [lo,hi) range of all three, sweep scratch is shared by position, and sibling
// subtrees are built by parallel tasks.  All arithmetic that decides the tree is IEEE binary64 in the
// reference's operation order (JS numbers are doubles), so split choices are identical:
//   cost(i) = 1 + (SAfront_i / SAparent) * (i+1) + (SAback_i / SAparent) * (n-1-i)        bvh.js:189
// where the back box still contains triangle i (the reference's off-by-one), first strict minimum over
// axis 0,1,2 and i ascending wins (bvh.js:190), leaves are ranges of <= maxTris (bvh.js:22) listed in
// x-sorted order (bvh.js:156-161).
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <chrono>
#include <atomic>
#include <future>
#include <thread>
#include <vector>

#include "../../include/fspt_b200.h"
#include "bvh_sah.h"

namespace {

struct BuildNode { Aabb box; int32_t left, right, lo, hi; };  // left < 0 => leaf over idx[0][lo,hi)

struct Ctx {
  const Aabb* tb;             // per-triangle boxes seen by the presorts and the SAH sweeps (Triangle.boundingBox)
  const Aabb* nb;             // per-triangle boxes of the current vertices (node boxes, BoundingBox.addNode)
  int32_t* idx[3];            // centroid-sorted triangle ids, partitioned in place
  int32_t* tmp[2];            // partition scratch (one per concurrently partitioned axis), indexed by position
  double* sback[3];           // suffix surface areas per axis, indexed by position
  uint8_t* side;              // per-triangle "goes left" flag
  std::vector<BuildNode> nodes;
  std::atomic<int32_t> n_nodes{0};
  std::atomic<int32_t> depth{0};
  std::atomic<int> failed{0};
  std::atomic<int> tasks_free{0};
  int max_tris;
};

template <class F>
void run_parallel(int n_threads, int n_items, F fn) {
  const int helpers = std::max(0, std::min(n_threads, n_items) - 1);
  std::atomic<int> next(0);
  auto work = [&]() { for (;;) { const int k = next.fetch_add(1); if (k >= n_items) break; fn(k); } };
  std::vector<std::thread> th;
  for (int i = 0; i < helpers; ++i) th.emplace_back(work);
  work();
  for (auto& t : th) t.join();
}

// Intra-node parallelism for the few huge nodes at the top of the tree (below them, sibling subtrees are the
// parallelism): up to `want` helper threads are borrowed from the same budget the subtree tasks use.
int grab(Ctx& c, int want) {
  int avail = c.tasks_free.load();
  for (;;) {
    const int take = std::min(avail, want);
    if (take <= 0) return 0;
    if (c.tasks_free.compare_exchange_weak(avail, avail - take)) return take;
  }
}
template <class F>
void par_items(Ctx& c, int n_items, F fn) {
  const int helpers = n_items > 1 ? grab(c, n_items - 1) : 0;
  if (helpers == 0) { for (int k = 0; k < n_items; ++k) fn(k); return; }
  std::atomic<int> next(0);
  auto work = [&]() { for (;;) { const int k = next.fetch_add(1); if (k >= n_items) break; fn(k); } };
  std::vector<std::thread> th;
  for (int i = 0; i < helpers; ++i) th.emplace_back(work);
  work();
  for (auto& t : th) t.join();
  c.tasks_free.fetch_add(helpers);
}
constexpr int32_t kParNode = 1 << 17;   // nodes at least this large are processed in chunks by several threads
constexpr int32_t kChunk = 1 << 15;

// Node.setSplit (bvh.js:168-197) for a huge node: min/max are exact and associative (incl. the signed-zero rule), so the
// front/back boxes of every position can be produced chunk by chunk from the unions of the chunks before/after it --
// the same doubles as the sequential sweep, hence the same costs and, merging in (axis, position) order with strict <,
// the same first minimum.
void split_parallel(Ctx& c, int32_t lo, int32_t hi, double parent, double& best, int& best_axis, int32_t& best_i) {
  const int32_t n = hi - lo;
  const int K = (int)std::min<int64_t>(64, ((int64_t)n + kChunk - 1) / kChunk);
  auto c0 = [&](int k) { return lo + (int32_t)((int64_t)n * k / K); };
  std::vector<Aabb> cbox((size_t)3 * K), pre((size_t)3 * K), suf((size_t)3 * K);
  par_items(c, 3 * K, [&](int item) {
    const int axis = item / K, k = item % K;
    const int32_t* ix = c.idx[axis];
    Aabb bb; bb.reset();
    for (int32_t i = c0(k); i < c0(k + 1); ++i) bb.grow(c.tb[ix[i]]);
    cbox[item] = bb;
  });
  for (int axis = 0; axis < 3; ++axis) {
    Aabb bb; bb.reset();
    for (int k = 0; k < K; ++k) { pre[axis * K + k] = bb; bb.grow(cbox[axis * K + k]); }
    bb.reset();
    for (int k = K - 1; k >= 0; --k) { suf[axis * K + k] = bb; bb.grow(cbox[axis * K + k]); }
  }
  std::vector<double> cbest((size_t)3 * K, INFINITY);
  std::vector<int32_t> cbest_i((size_t)3 * K, -1);
  par_items(c, 3 * K, [&](int item) {
    const int axis = item / K, k = item % K;
    const int32_t* ix = c.idx[axis];
    double* sback = c.sback[axis];
    const int32_t a = c0(k), b = c0(k + 1);
    Aabb bb = suf[item];
    for (int32_t i = b - 1; i >= a; --i) { bb.grow(c.tb[ix[i]]); sback[i] = bb.area(); }
    bb = pre[item];
    double bst = INFINITY; int32_t bi = -1;
    for (int32_t i = a; i < b; ++i) {
      bb.grow(c.tb[ix[i]]);
      const double sAf = bb.area(), sAb = sback[i];
      const int32_t kk = i - lo;
      const double cost = sah_cost(sAf, sAb, parent, kk, n);
      if (cost < bst) { bst = cost; bi = kk + 1; }
    }
    cbest[item] = bst; cbest_i[item] = bi;
  });
  for (int item = 0; item < 3 * K; ++item)
    if (cbest[item] < best) { best = cbest[item]; best_i = cbest_i[item]; best_axis = item / K; }
}

int32_t build(Ctx& c, int32_t lo, int32_t hi, int d) {
  int32_t self = c.n_nodes.fetch_add(1);
  BuildNode nd;
  nd.lo = lo; nd.hi = hi; nd.left = nd.right = -1;
  int prev = c.depth.load();
  while (d > prev && !c.depth.compare_exchange_weak(prev, d)) {}
  const int32_t n = hi - lo;
  nd.box.reset();
  const bool big = n >= kParNode && c.tasks_free.load() > 0;  // helpers available (otherwise the plain sweep is cheaper)
  if (!big) {
    for (int32_t i = lo; i < hi; ++i) nd.box.grow(c.nb[c.idx[0][i]]);  // BoundingBox.addNode, bvh.js:122-128
  } else {
    const int K = (int)std::min<int64_t>(64, ((int64_t)n + kChunk - 1) / kChunk);
    std::vector<Aabb> part((size_t)K);
    par_items(c, K, [&](int k) {
      Aabb bb; bb.reset();
      const int32_t a = lo + (int32_t)((int64_t)n * k / K), b = lo + (int32_t)((int64_t)n * (k + 1) / K);
      for (int32_t i = a; i < b; ++i) bb.grow(c.nb[c.idx[0][i]]);
      part[k] = bb;
    });
    for (int k = 0; k < K; ++k) nd.box.grow(part[k]);
  }
  if (n <= c.max_tris) { c.nodes[self] = nd; return self; }          // bvh.js:22 (split of a leaf is unused)
  // Node.setSplit, bvh.js:168-197
  double best = INFINITY;
  int best_axis = -1; int32_t best_i = -1;
  const double parent = nd.box.area();
  if (big) split_parallel(c, lo, hi, parent, best, best_axis, best_i);
  else for (int axis = 0; axis < 3; ++axis) {
    const int32_t* ix = c.idx[axis];
    double* sback = c.sback[0];
    Aabb bb; bb.reset();
    for (int32_t i = hi - 1; i >= lo; --i) { bb.grow(c.tb[ix[i]]); sback[i] = bb.area(); }
    bb.reset();
    for (int32_t i = lo; i < hi; ++i) {
      bb.grow(c.tb[ix[i]]);
      const double sAf = bb.area(), sAb = sback[i];
      const int32_t k = i - lo;
      const double cost = sah_cost(sAf, sAb, parent, k, n);
      if (cost < best) { best = cost; best_i = k + 1; best_axis = axis; }
    }
  }
  if (best_axis < 0 || best_i >= n || d > 4000) {  // JS: TypeError on undefined axis / unbounded recursion
    c.failed.store(1);
    c.nodes[self] = nd;
    return self;
  }
  // _constructCachedIndexList, bvh.js:52-76: stable partition of the other two axes
  const int32_t mid = lo + best_i;
  for (int32_t i = lo; i < hi; ++i) c.side[c.idx[best_axis][i]] = (i < mid);
  auto partition_axis = [&](int which) {  // which = 0, 1: the two axes other than best_axis, each with its own scratch
    const int axis = (best_axis + 1 + which) % 3;
    int32_t* ix = c.idx[axis];
    int32_t* tmp = c.tmp[which];
    int32_t l = lo, r = 0;
    for (int32_t i = lo; i < hi; ++i) { int32_t t = ix[i]; if (c.side[t]) ix[l++] = t; else tmp[lo + r++] = t; }
    memcpy(ix + l, tmp + lo, sizeof(int32_t) * (size_t)r);
  };
  if (big) par_items(c, 2, partition_axis);
  else { partition_axis(0); partition_axis(1); }
  int32_t L, R;
  bool spawn = false;
  if (n > 32768) {  // sibling subtrees touch disjoint ranges / triangles: build them concurrently
    int avail = c.tasks_free.load();
    while (avail > 0 && !c.tasks_free.compare_exchange_weak(avail, avail - 1)) {}
    spawn = avail > 0;
  }
  if (spawn) {
    auto fut = std::async(std::launch::async, [&c, lo, mid, d]() { return build(c, lo, mid, d + 1); });
    R = build(c, mid, hi, d + 1);
    L = fut.get();
    c.tasks_free.fetch_add(1);
  } else {
    L = build(c, lo, mid, d + 1);
    R = build(c, mid, hi, d + 1);
  }
  nd.left = L; nd.right = R;
  c.nodes[self] = nd;
  return self;
}

// serializeTree (bvh.js:33-50) + flatten (main.js:366-392): pre-order, iterative
void flatten(const Ctx& c, int32_t root, float* out, int32_t* order, int32_t* n_out) {
  struct Item { int32_t node; int32_t parent_slot; int which; };
  std::vector<Item> st;
  st.push_back({root, -1, 0});
  int32_t n = 0, tri = 0;
  while (!st.empty()) {
    Item it = st.back(); st.pop_back();
    const BuildNode& b = c.nodes[it.node];
    const int32_t self = n++;
    float* p = out + (size_t)self * 9;
    int32_t l = 0, r = 0, t = -1;  // leaf: left/right undefined -> Int32Array 0 (main.js:275)
    if (b.left < 0) {
      t = tri;                      // trianglesBuffer.length/9 (main.js:369)
      for (int32_t i = b.lo; i < b.hi; ++i) order[tri++] = c.idx[0][i];
    }
    memcpy(p + 0, &l, 4); memcpy(p + 1, &r, 4); memcpy(p + 2, &t, 4);  // maskBVHBuffer, main.js:272-282
    for (int k = 0; k < 3; ++k) { p[3 + k] = (float)b.box.mn[k]; p[6 + k] = (float)b.box.mx[k]; }
    if (it.parent_slot >= 0) memcpy(out + (size_t)it.parent_slot * 9 + it.which, &self, 4);
    if (b.left >= 0) {  // right pushed first so the left subtree is numbered first (pre-order)
      st.push_back({b.right, self, 1});
      st.push_back({b.left, self, 0});
    }
  }
  *n_out = n;
}

}  // namespace

extern "C" int fspt_bvh_build(const double* verts, int32_t n_tris, int32_t max_tris, float* nodes_out,
                              int32_t* order_out, int32_t* n_nodes_out, int32_t* depth_out, int32_t n_threads) {
  return fspt_bvh_build2(verts, nullptr, n_tris, max_tris, nodes_out, order_out, n_nodes_out, depth_out, n_threads);
}

// box_verts != NULL reproduces `scene.normalize` (main.js:337-348): Triangle.boundingBox is computed when the
// triangle is created (bvh.js:208) and NOT refreshed when normalize rescales the vertices, so the presorts and
// the SAH sweeps see the old boxes (box_verts) while node boxes are built from the new vertices (verts).
extern "C" int fspt_bvh_build2(const double* verts, const double* box_verts, int32_t n_tris, int32_t max_tris,
                               float* nodes_out, int32_t* order_out, int32_t* n_nodes_out, int32_t* depth_out,
                               int32_t n_threads) {
  if (!verts || !nodes_out || !order_out || n_tris <= 0 || max_tris <= 0) return FSPT_E_INVALID;
  const bool timing = getenv("FSPT_TIMING") != nullptr;
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!timing) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[fspt bvh] %-24s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - t_prev).count());
    t_prev = now;
  };
  const double* bv = box_verts ? box_verts : verts;
  std::vector<Aabb> tb((size_t)n_tris), nb;
  if (box_verts) nb.resize((size_t)n_tris);
  std::vector<double> cen[3];
  for (int a = 0; a < 3; ++a) cen[a].resize((size_t)n_tris);
  if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
  n_threads = std::max(1, n_threads);
  std::atomic<int> bad(0);
  const int box_chunks = (int)std::min<int64_t>(256, ((int64_t)n_tris + 65535) / 65536);
  run_parallel(n_threads, box_chunks, [&](int ch) {
    const int32_t i0 = (int32_t)((int64_t)n_tris * ch / box_chunks), i1 = (int32_t)((int64_t)n_tris * (ch + 1) / box_chunks);
    for (int32_t i = i0; i < i1; ++i) {  // Triangle.boundingBox, bvh.js:208
      Aabb& b = tb[i]; b.reset();
      for (int v = 0; v < 3; ++v)
        for (int k = 0; k < 3; ++k) {
          double x = bv[(size_t)i * 9 + v * 3 + k];
          if (!finite_coord(x)) { bad.store(1); return; }
          b.add_point(x, k);
        }
      for (int k = 0; k < 3; ++k) cen[k][i] = b.centroid(k);
      if (box_verts) {
        Aabb& n = nb[i]; n.reset();
        for (int v = 0; v < 3; ++v)
          for (int k = 0; k < 3; ++k) {
            double x = verts[(size_t)i * 9 + v * 3 + k];
            if (!finite_coord(x)) { bad.store(1); return; }
            n.add_point(x, k);
          }
      }
    }
  });
  if (bad.load()) return FSPT_E_INVALID;
  lap("boxes + centroids");
  std::vector<int32_t> ix[3], tmp[2];
  for (auto& t : tmp) t.resize((size_t)n_tris);
  std::vector<double> sback[3];
  sback[0].resize((size_t)n_tris);
  if (n_tris >= kParNode) { sback[1].resize((size_t)n_tris); sback[2].resize((size_t)n_tris); }
  std::vector<uint8_t> side((size_t)n_tris);
  {
    // _sortIndices x3 (bvh.js:78-90): stable, by centroid.  Large inputs: every axis is cut into runs that are
    // stable-sorted concurrently and then merged pairwise (a stable merge of adjacent runs yields the one stable order).
    const int P = n_tris >= kParNode ? 8 : 1;
    auto run0 = [&](int r) { return (int32_t)((int64_t)n_tris * r / P); };
    for (int a = 0; a < 3; ++a) ix[a].resize((size_t)n_tris);
    run_parallel(n_threads, 3 * P, [&](int item) {
      const int a = item / P, r = item % P;
      const double* cc = cen[a].data();
      int32_t* v = ix[a].data();
      for (int32_t i = run0(r); i < run0(r + 1); ++i) v[i] = i;
      std::stable_sort(v + run0(r), v + run0(r + 1), [cc](int32_t p, int32_t q) { return cc[p] < cc[q]; });
    });
    for (int width = 1; width < P; width *= 2) {
      const int pairs = P / (2 * width);
      run_parallel(n_threads, 3 * pairs, [&](int item) {
        const int a = item / pairs, j = item % pairs;
        const double* cc = cen[a].data();
        int32_t* v = ix[a].data();
        std::inplace_merge(v + run0(2 * j * width), v + run0((2 * j + 1) * width), v + run0((2 * j + 2) * width),
                           [cc](int32_t p, int32_t q) { return cc[p] < cc[q]; });
      });
    }
  }
  lap("presort x3");
  Ctx c;
  c.tb = tb.data();
  c.nb = box_verts ? nb.data() : tb.data();
  for (int a = 0; a < 3; ++a) c.idx[a] = ix[a].data();
  c.tmp[0] = tmp[0].data(); c.tmp[1] = tmp[1].data();
  for (int a = 0; a < 3; ++a) c.sback[a] = sback[a].empty() ? sback[0].data() : sback[a].data();
  c.side = side.data();
  c.nodes.resize((size_t)2 * n_tris + 1);
  c.max_tris = max_tris;
  c.tasks_free.store(n_threads > 1 ? n_threads - 1 : 0);
  int32_t root = build(c, 0, n_tris, 0);
  lap("build");
  if (c.failed.load()) return FSPT_E_LIMIT;
  int32_t n = 0;
  flatten(c, root, nodes_out, order_out, &n);
  lap("flatten");
  if (n_nodes_out) *n_nodes_out = n;
  if (depth_out) *depth_out = c.depth.load();
  return FSPT_OK;
}

// ProcessEnvRadiance (env_sampler.js:1-74).  Same boxes as the JavaScript: region sums are accumulated in the
// reference's own order (x-major double additions over the first half of every box, env_sampler.js:36-41), because the
// split decisions compare those rounded sums -- a summed-area table would change them in the last place.
extern "C" int fspt_env_bins(const uint8_t* data, int32_t width, int32_t height, uint16_t* bins_out,
                             int32_t capacity, int32_t* n_u16_out) {
  if (!data || !bins_out || width <= 0 || height <= 0 || capacity < 4) return FSPT_E_INVALID;
  // luminance per texel in double, env_sampler.js:14-22
  std::vector<double> lum((size_t)width * height);
  double total = 0, brightest = 0;
  for (int y = 0; y < height; ++y)
    for (int x = 0; x < width; ++x) {
      const uint8_t* p = data + ((size_t)y * width + x) * 4;
      double power = ldexp(1.0, (int)p[3] - 128);  // Math.pow(2, a-128) is exact
      double r = power * p[0] / 255.0, g = power * p[1] / 255.0, b = power * p[2] / 255.0;
      double l = 0.2126 * r + 0.7152 * g + 0.0722 * b;
      lum[(size_t)y * width + x] = l;
      if (l > brightest) brightest = l;
      total += l;
    }
  const double minRadiance = std::max(total / 64, brightest / 2);
  std::vector<double> boxes;
  struct Frame { double radiance, x0, y0, x1, y1; };
  std::vector<Frame> stack;
  stack.push_back({total, 0, 0, (double)width, (double)height});
  auto lumAt = [&](double x, double y) -> double {  // data[fractional index] is undefined -> NaN in JS
    if (x != floor(x) || y != floor(y)) return NAN;
    size_t off = (size_t)y * (size_t)width + (size_t)x;
    if (off >= lum.size()) return NAN;
    return lum[off];
  };
  while (!stack.empty()) {  // biSplit, env_sampler.js:26-50 (explicit stack, same DFS emission order)
    Frame f = stack.back(); stack.pop_back();
    if ((int64_t)boxes.size() + 4 > capacity) break;
    if (f.radiance <= minRadiance || (f.y1 - f.y0) * (f.x1 - f.x0) < 2) {
      boxes.push_back(f.x0); boxes.push_back(f.y0); boxes.push_back(f.x1); boxes.push_back(f.y1);
      continue;
    }
    double sub = 0;
    bool vert = f.x1 - f.x0 > f.y1 - f.y0;
    double xs = f.x1, ys = (f.y1 - f.y0) / 2 + f.y0;
    if (vert) { xs = (f.x1 - f.x0) / 2 + f.x0; ys = f.y1; }
    for (double x = f.x0; x < xs; x++)
      for (double y = f.y0; y < ys; y++) sub += lumAt(x, y);
    // second half pushed first so the first half is processed (and emitted) first
    if (vert) stack.push_back({f.radiance - sub, xs, f.y0, f.x1, f.y1});
    else stack.push_back({f.radiance - sub, f.x0, ys, f.x1, f.y1});
    stack.push_back({sub, f.x0, f.y0, xs, ys});
  }
  int n = (int)boxes.size();
  for (int i = 0; i < n; ++i) {  // new Uint16Array(boxes): ToUint16
    double v = boxes[i];
    if (v != v || isinf(v)) { bins_out[i] = 0; continue; }
    double tr = v < 0 ? ceil(v) : floor(v);
    bins_out[i] = (uint16_t)(uint64_t)(int64_t)fmod(tr, 65536.0);
  }
  if (n_u16_out) *n_u16_out = n;
  return FSPT_OK;
}

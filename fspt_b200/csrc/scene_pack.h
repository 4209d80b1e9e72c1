// scene_pack.h -- host side of fspt_scene_upload that has nothing to do with CUDA: the pre-passes over the reference-layout
// arrays (interior-record numbering, material ids, depth / tree check) and the builders of the device records
// (Node64, Tri48, ShadeRec; device_common.cuh / DESIGN.md section 3).  Plain C++ on top of host_pool.h, so that the CPU
// suite can run it without a GPU (fspt_debug_pack_scene, tests/test_scene_pack.py).
#pragma once
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <array>
#include <atomic>
#include <map>
#include <string>
#include <vector>

#include "../../include/fspt_b200.h"
#include "host_pool.h"

#ifndef FSPT_STACK
#define FSPT_STACK 64 /* tracer.fs:368 */
#endif

struct ScenePrepass {
  std::vector<int32_t> ref;          // child reference of reference node i: >= 0 interior record, < 0 ~first triangle
  std::vector<int32_t> interior_of;  // reference node index of interior record k
  std::vector<int32_t> mat_id;       // per triangle: index into mats
  std::vector<std::array<int, 4>> mats;  // distinct quadruples of atlas layers (diffuse, emission, metallic-roughness, normal)
  bool dielectric = false;           // any triangle with materials[10] >= 0 (tracer.fs:481)
  int max_depth = 0;
  std::string error;                 // set when the return value is not FSPT_OK
  size_t NI() const { return interior_of.size(); }
};

inline int32_t scene_node_bits(const fspt_scene_desc* s, int node, int k) {
  int32_t v;
  memcpy(&v, s->bvh + (size_t)node * 9 + k, 4);
  return v;
}

// Two parallel regions around a short serial step.
// Nodes: reference node i = [left, right, triIndex | min | max] -> child references; interior nodes are numbered in
// node order (count per chunk, prefix sum over the chunks, assign).
// Triangles: materials = distinct quadruples of atlas layers, tracer.fs:453-456, numbered in order of first appearance
// (local numbering per chunk, serial merge of the few keys, then the chunks rewrite their ids if the merge changed any).
// Depth / stack bound check (the reference has int stack[64], tracer.fs:368): the top of the tree is walked serially
// until there are a few subtrees per worker, each subtree is then an item (iterative DFS).  Child indices out of range
// end a walk silently; pack_node_chunk reports them.
inline int scene_prepass(HostPool& pool, int hw, const fspt_scene_desc* s, ScenePrepass& P) {
  const int N = s->n_nodes, T = s->n_triangles;
  auto ibits = [&](int node, int k) { return scene_node_bits(s, node, k); };
  auto fail = [&](int code, const char* fmt, int a0, int a1) {
    char buf[192];
    snprintf(buf, sizeof buf, fmt, a0, a1);
    P.error = buf;
    return code;
  };
  P.ref.assign((size_t)N, 0);
  P.mat_id.assign((size_t)T, 0);
  P.mats.clear();
  P.dielectric = false;
  const int PRE_CHUNK = 8192;
  const int n_nchunks = (N + PRE_CHUNK - 1) / PRE_CHUNK, n_tchunks = (T + PRE_CHUNK - 1) / PRE_CHUNK;
  std::vector<int> chunk_interiors((size_t)n_nchunks + 1, 0);
  std::atomic<int> bad_node(-1);
  std::vector<std::vector<std::array<int, 4>>> local_keys((size_t)n_tchunks);
  std::vector<int> local_diel((size_t)n_tchunks, 0);
  auto layer_of = [&](float lf) {  // texture(texArray, vec3(uv, layer)): layer = clamp(floor(l + 0.5), 0, d - 1)
    float f = floorf(lf + 0.5f);
    if (!(f >= -1.0e9f && f <= 1.0e9f)) f = 0.0f;
    long long q = (long long)f;
    return (int)(q < 0 ? 0 : (q >= s->atlas_layers ? s->atlas_layers - 1 : q));
  };
  struct Sub { int node, depth; };
  std::vector<Sub> subtrees;
  int top_depth = 0;
  size_t top_visited = 0;
  {
    std::vector<Sub> frontier{{0, 1}}, next;
    while (!frontier.empty() && frontier.size() < (size_t)(8 * hw) && top_visited <= (size_t)N) {
      next.clear();
      for (const Sub& f : frontier) {
        ++top_visited;
        top_depth = std::max(top_depth, f.depth);
        if (ibits(f.node, 2) > -1) continue;
        const int32_t l = ibits(f.node, 0), r = ibits(f.node, 1);
        if (l < 0 || l >= N || r < 0 || r >= N) continue;
        next.push_back({l, f.depth + 1});
        next.push_back({r, f.depth + 1});
      }
      frontier.swap(next);
    }
    subtrees.swap(frontier);
  }
  const int n_sub = (int)subtrees.size();
  std::vector<int> sub_depth((size_t)n_sub, 0);
  std::vector<size_t> sub_visited((size_t)n_sub, 0);
  pool.run(n_nchunks + n_tchunks + n_sub, hw, [&](int item) {
    if (item >= n_nchunks + n_tchunks) {
      const int k = item - n_nchunks - n_tchunks;
      std::vector<Sub> st;
      st.reserve(128);
      st.push_back(subtrees[k]);
      int max_depth = 0;
      size_t visited = 0;
      while (!st.empty()) {
        const Sub n = st.back(); st.pop_back();
        if (++visited > (size_t)N) break;  // more visits than nodes: not a tree
        max_depth = std::max(max_depth, n.depth);
        if (ibits(n.node, 2) > -1) continue;
        const int32_t l = ibits(n.node, 0), r = ibits(n.node, 1);
        if (l < 0 || l >= N || r < 0 || r >= N) continue;
        st.push_back({l, n.depth + 1});
        st.push_back({r, n.depth + 1});
      }
      sub_depth[k] = max_depth; sub_visited[k] = visited;
      return;
    }
    if (item < n_nchunks) {
      const int ch = item, i1 = std::min(N, (ch + 1) * PRE_CHUNK);
      int n_int = 0;
      for (int i = ch * PRE_CHUNK; i < i1; ++i) {
        const int32_t tri = ibits(i, 2);
        if (tri > -1) {  // `current.triangles > -1`, tracer.fs:379
          if (tri >= T) { int exp = -1; bad_node.compare_exchange_strong(exp, i); }
        } else {
          ++n_int;
        }
      }
      chunk_interiors[ch + 1] = n_int;
      return;
    }
    const int ch = item - n_nchunks, t0 = ch * PRE_CHUNK, t1 = std::min(T, (ch + 1) * PRE_CHUNK);
    std::map<std::array<int, 4>, int> ids;
    std::vector<std::array<int, 4>>& keys = local_keys[ch];
    std::array<int, 4> last = {-1, -1, -1, -1};
    int last_id = -1, diel = 0;
    for (int t = t0; t < t1; ++t) {
      const float* o = s->materials + (size_t)t * 12;
      if (o[10] >= 0.0f) diel = 1;
      if (t > t0 && memcmp(o, o - 12, 16) == 0) { P.mat_id[t] = last_id; continue; }  // same four layer floats as the previous triangle
      const std::array<int, 4> key = {layer_of(o[0]), layer_of(o[1]), layer_of(o[3]), layer_of(o[2])};
      if (key != last) {
        auto it = ids.find(key);
        if (it == ids.end()) { it = ids.emplace(key, (int)keys.size()).first; keys.push_back(key); }
        last = key; last_id = it->second;
      }
      P.mat_id[t] = last_id;
    }
    local_diel[ch] = diel;
  });
  if (bad_node.load() >= 0)
    return fail(FSPT_E_INVALID, "node %d: triangle index %d out of range", bad_node.load(), ibits(bad_node.load(), 2));
  {
    int max_depth = top_depth;
    size_t visited = top_visited;
    for (int k = 0; k < n_sub; ++k) { max_depth = std::max(max_depth, sub_depth[k]); visited += sub_visited[k]; }
    if (visited > (size_t)N) return fail(FSPT_E_INVALID, "BVH is not a tree (cycle or shared node)", 0, 0);
    // max_depth counts the nodes on the longest root-to-leaf path.  The walk down it defers at most one child per interior
    // node (max_depth - 1 entries) on top of the sentinel, so a tree of FSPT_STACK levels fills the stack exactly.
    if (max_depth > FSPT_STACK)
      return fail(FSPT_E_LIMIT, "BVH of %d levels exceeds the traversal stack (at most %d levels, tracer.fs:368)", max_depth,
                  FSPT_STACK);
    P.max_depth = max_depth;
  }
  for (int ch = 0; ch < n_nchunks; ++ch) chunk_interiors[ch + 1] += chunk_interiors[ch];
  P.interior_of.assign((size_t)chunk_interiors[n_nchunks], 0);
  std::vector<std::vector<int>> remap((size_t)n_tchunks);
  bool identity = true;
  {
    std::map<std::array<int, 4>, int> ids;
    for (int ch = 0; ch < n_tchunks; ++ch) {
      P.dielectric = P.dielectric || local_diel[ch];
      remap[ch].resize(local_keys[ch].size());
      for (size_t k = 0; k < local_keys[ch].size(); ++k) {
        auto it = ids.find(local_keys[ch][k]);
        if (it == ids.end()) { it = ids.emplace(local_keys[ch][k], (int)P.mats.size()).first; P.mats.push_back(local_keys[ch][k]); }
        remap[ch][k] = it->second;
        identity = identity && it->second == (int)k;
      }
    }
  }
  pool.run(n_nchunks + (identity ? 0 : n_tchunks), hw, [&](int item) {
    if (item < n_nchunks) {
      const int ch = item, i1 = std::min(N, (ch + 1) * PRE_CHUNK);
      int k = chunk_interiors[ch];
      for (int i = ch * PRE_CHUNK; i < i1; ++i) {
        const int32_t tri = ibits(i, 2);
        if (tri > -1) P.ref[i] = ~tri;
        else { P.ref[i] = k; P.interior_of[(size_t)k++] = i; }
      }
      return;
    }
    const int ch = item - n_nchunks, t1 = std::min(T, (ch + 1) * PRE_CHUNK);
    const std::vector<int>& r = remap[ch];
    for (int t = ch * PRE_CHUNK; t < t1; ++t) P.mat_id[t] = r[P.mat_id[t]];
  });
  return FSPT_OK;
}

// Node64 for interior records [k0, k1): (left, right) pairs per component -- the operand layout of the packed f32x2 slab
// test -- then the two child references.  `out` receives (k1 - k0) * 16 floats (one zeroed record when the tree has no
// interior node at all).  Returns the reference index of the first node with a bad child index, or -1.
inline int pack_node_chunk(const fspt_scene_desc* s, const ScenePrepass& P, size_t k0, size_t k1, float* out, int* bad_l, int* bad_r) {
  const int N = s->n_nodes;
  int bad = -1;
  if (P.NI() == 0) memset(out, 0, 64);
  for (size_t k = k0; k < k1; ++k) {
    const int i = P.interior_of[k];
    const int32_t l = scene_node_bits(s, i, 0), r = scene_node_bits(s, i, 1);
    float* o = out + (k - k0) * 16;
    if (l < 0 || l >= N || r < 0 || r >= N || l == i || r == i) {
      if (bad < 0) { bad = i; *bad_l = l; *bad_r = r; }
      memset(o, 0, 64);
      continue;
    }
    const float* lb = s->bvh + (size_t)l * 9 + 3;
    const float* rb = s->bvh + (size_t)r * 9 + 3;
    for (int q = 0; q < 6; ++q) { o[2 * q] = lb[q]; o[2 * q + 1] = rb[q]; }
    const int32_t lr = P.ref[l], rr = P.ref[r];
    memcpy(o + 12, &lr, 4); memcpy(o + 13, &rr, 4);
    o[14] = o[15] = 0.0f;
  }
  return bad;
}

// Tri48 for triangles [t0, t1) (t1 <= T + 3: the LEAF_SIZE-1 padBuffer-style (-1,-1,-1) tail records, main.js:143-154) and
// ShadeRec for [t0, min(t1, T)).  Tri48 = v1 | e1 | e2 (the two subtractions of tracer.fs:301-302 as single f32
// operations) | pad; ShadeRec = material (12) | uvs (6) | material id | pad | normals (27) | pad.
inline void pack_tri_chunk(const fspt_scene_desc* s, const ScenePrepass& P, int t0, int t1, float* tris, float* shade) {
  const int T = s->n_triangles;
  for (int t = t0; t < t1; ++t) {
    float* o = tris + (size_t)(t - t0) * 12;
    float v[9];
    if (t < T) memcpy(v, s->triangles + (size_t)t * 9, sizeof v);
    else for (float& x : v) x = -1.0f;
    o[0] = v[0]; o[1] = v[1]; o[2] = v[2];
    volatile float e;  // keep these as single f32 subtractions
    e = v[3] - v[0]; o[3] = e; e = v[4] - v[1]; o[4] = e; e = v[5] - v[2]; o[5] = e;
    e = v[6] - v[0]; o[6] = e; e = v[7] - v[1]; o[7] = e; e = v[8] - v[2]; o[8] = e;
    o[9] = o[10] = o[11] = 0.0f;
    if (t >= T) continue;
    float* h = shade + (size_t)(t - t0) * 48;
    memcpy(h, s->materials + (size_t)t * 12, 48);
    memcpy(h + 12, s->uvs + (size_t)t * 6, 24);
    memcpy(h + 18, &P.mat_id[t], 4);  // material id in the record's padding
    h[19] = 0.0f;
    memcpy(h + 20, s->normals + (size_t)t * 27, 108);
    h[47] = 0.0f;
  }
}

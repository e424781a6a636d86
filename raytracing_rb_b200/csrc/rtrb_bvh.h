// rtrb_bvh.h — host-side build of the sphere BVH used by the FAST64 FP32 filter (SURVEY.md 8f rank 1:
// the reference's own TODO "速度优化(xx树)", README.md:13).
//
// The tree only accelerates the FILTER: it decides which spheres get the FP32 line test and, if they
// survive, the exact FP64 test.  It can therefore never change a result as long as it is
// conservative, i.e. every sphere the strict scan (world.rb:44-57) could accept is reached.  Boxes are
// the exact FP64 sphere bounds rounded OUTWARD to FP32; the per-ray error margin E is added at
// traversal time (rtrb_trace_fast.cuh).  Ties and ordering are untouched: survivors are still
// compared on (distance, world index) / subtracted in world-index order.
#pragma once
#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <vector>

struct BvhNode {        // 64 B: both child boxes live in the parent, one fetch decides both
  float lo0[3], hi0[3];
  float lo1[3], hi1[3];
  int32_t child0, child1;  // >= 0: node index; < 0: leaf, ~child = first | (count << 20)
  int32_t pad0, pad1;
};

struct BvhBuildSphere {
  double c[3], r;
  int32_t world_index;
  int32_t bound_only = 0;  // bounding sphere of a box (rtrb_types.h, cull_sph)
};

namespace rtrb_bvh {

struct Box { float lo[3], hi[3]; };

inline float round_down(double v) { float f = (float)v; return (double)f > v ? nextafterf(f, -INFINITY) : f; }
inline float round_up(double v) { float f = (float)v; return (double)f < v ? nextafterf(f, INFINITY) : f; }

inline Box empty_box() { Box b; for (int k = 0; k < 3; ++k) { b.lo[k] = INFINITY; b.hi[k] = -INFINITY; } return b; }
inline void grow(Box& b, const BvhBuildSphere& s) {
  for (int k = 0; k < 3; ++k) {
    b.lo[k] = std::min(b.lo[k], round_down(s.c[k] - fabs(s.r)));
    b.hi[k] = std::max(b.hi[k], round_up(s.c[k] + fabs(s.r)));
  }
}

constexpr int kLeafSize = 4;

// Recursively builds over order[first, first+count); returns the child reference for this subtree and its box.
inline int32_t build(std::vector<BvhNode>& nodes, std::vector<BvhBuildSphere>& sph, int first, int count, Box* box_out) {
  Box box = empty_box();
  for (int i = first; i < first + count; ++i) grow(box, sph[i]);
  *box_out = box;
  if (count <= kLeafSize) return ~(int32_t)((uint32_t)first | ((uint32_t)count << 20));
  // split at the median of the widest centroid axis
  double cmin[3] = {INFINITY, INFINITY, INFINITY}, cmax[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = first; i < first + count; ++i)
    for (int k = 0; k < 3; ++k) { cmin[k] = std::min(cmin[k], sph[i].c[k]); cmax[k] = std::max(cmax[k], sph[i].c[k]); }
  int axis = 0;
  for (int k = 1; k < 3; ++k) if (cmax[k] - cmin[k] > cmax[axis] - cmin[axis]) axis = k;
  int mid = first + count / 2;
  std::nth_element(sph.begin() + first, sph.begin() + mid, sph.begin() + first + count,
                   [axis](const BvhBuildSphere& a, const BvhBuildSphere& b) {
                     return a.c[axis] < b.c[axis] || (a.c[axis] == b.c[axis] && a.world_index < b.world_index);
                   });
  int me = (int)nodes.size();
  nodes.emplace_back();
  Box b0, b1;
  int32_t c0 = build(nodes, sph, first, mid - first, &b0);
  int32_t c1 = build(nodes, sph, mid, first + count - mid, &b1);
  BvhNode& n = nodes[me];
  for (int k = 0; k < 3; ++k) { n.lo0[k] = b0.lo[k]; n.hi0[k] = b0.hi[k]; n.lo1[k] = b1.lo[k]; n.hi1[k] = b1.hi[k]; }
  n.child0 = c0; n.child1 = c1; n.pad0 = n.pad1 = 0;
  return me;
}

// Reorders `sph` so that every leaf is a contiguous range and returns the node array; node 0 is the
// root.  With <= kLeafSize spheres the root is a node whose child0 is the single leaf and child1 is empty.
inline std::vector<BvhNode> build_tree(std::vector<BvhBuildSphere>& sph) {
  std::vector<BvhNode> nodes;
  if (sph.empty()) return nodes;
  nodes.reserve(sph.size());
  Box box;
  if ((int)sph.size() <= kLeafSize) {
    nodes.emplace_back();
    Box b0;
    int32_t c0 = build(nodes, sph, 0, (int)sph.size(), &b0);
    BvhNode& n = nodes[0];
    Box e = empty_box();
    for (int k = 0; k < 3; ++k) { n.lo0[k] = b0.lo[k]; n.hi0[k] = b0.hi[k]; n.lo1[k] = e.lo[k]; n.hi1[k] = e.hi[k]; }
    n.child0 = c0; n.child1 = ~(int32_t)0;  // empty leaf
    n.pad0 = n.pad1 = 0;
    return nodes;
  }
  build(nodes, sph, 0, (int)sph.size(), &box);
  return nodes;
}

}  // namespace rtrb_bvh

// bvh_sah.h -- the arithmetic that decides a bvh.js tree, shared by the host builder (bvh_builder.cpp, g++) and the
// device builder (bvh_device.cu, nvcc).  Both compile it with contraction off (-ffp-contract=off / --fmad=false), so every
// value below is the same IEEE binary64 result on either side and the two builders cannot drift apart.
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define FSPT_HD __host__ __device__ __forceinline__
#else
#define FSPT_HD inline
#endif

struct Aabb {
  double mn[3], mx[3];
  FSPT_HD void reset() { for (int k = 0; k < 3; ++k) { mn[k] = INFINITY; mx[k] = -INFINITY; } }
  // Math.min / Math.max (vector.js:55-61) incl. their signed-zero rule (-0 < +0); inputs are never NaN (checked)
  static FSPT_HD double lo(double a, double b) { return a < b ? a : (b < a ? b : (signbit(a) ? a : b)); }
  static FSPT_HD double hi(double a, double b) { return a < b ? b : (b < a ? a : (signbit(a) ? b : a)); }
  FSPT_HD void grow(const Aabb& b) {
    for (int k = 0; k < 3; ++k) { mn[k] = lo(mn[k], b.mn[k]); mx[k] = hi(mx[k], b.mx[k]); }
  }
  FSPT_HD void add_point(double x, int k) { mn[k] = lo(x, mn[k]); mx[k] = hi(x, mx[k]); }
  FSPT_HD double area() const {  // BoundingBox.getSurfaceArea, bvh.js:137-142
    double xl = mx[0] - mn[0], yl = mx[1] - mn[1], zl = mx[2] - mn[2];
    return (xl * yl + xl * zl + yl * zl) * 2;
  }
  FSPT_HD double centroid(int k) const { return (mn[k] + mx[k]) * 0.5; }  // bvh.js:130-135
};

// bvh.js:189: the cost of putting the first k+1 of n triangles in front (the back box still holds triangle k)
FSPT_HD double sah_cost(double sAf, double sAb, double parent, int32_t k, int32_t n) {
  return 1 + (sAf / parent) * 1 * (double)(k + 1) + (sAb / parent) * 1 * (double)(n - 1 - k);
}

// Finite coordinates only: bvh.js would build a tree from NaN / inf boxes that no traversal can use.
FSPT_HD bool finite_coord(double x) { return x == x && !isinf(x); }

// fp64 point/triangle geometry shared by the seed generator (seedgen.cu) and the point-to-mesh distance (mesh_dist.cu).
// Both files are compiled with -fmad=false: every product and sum below rounds on its own, in the order written, so a
// numpy restatement of the same expressions gives the same bits.
#pragma once
#include "common.cuh"

namespace sapcu {

struct V3 { double x, y, z; };
__device__ __forceinline__ V3 vsub(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ V3 vadd(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ V3 vmul(V3 a, double s) { return {a.x * s, a.y * s, a.z * s}; }
__device__ __forceinline__ V3 vdiv(V3 a, double s) { return {a.x / s, a.y / s, a.z / s}; }
__device__ __forceinline__ double vdot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ V3 vcross(V3 a, V3 b) {
  return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
__device__ __forceinline__ double vdist(V3 a, V3 b) {
  return sqrt((a.x - b.x) * (a.x - b.x) + (a.y - b.y) * (a.y - b.y) + (a.z - b.z) * (a.z - b.z));
}

// closest point on triangle abc to p -- dense.cpp:135-174, same branch order and operation order.
// Degenerate faces can reach a 0/0 and return NaN: with a == b != c and p beyond a in the direction of c (tnom > 0,
// tdenom > 0) the edge-ab branch divides snom * ab = 0 by snom + sdenom = 0; and whenever n == 0 (coincident or exactly
// collinear vertices) a point reaching the barycentric branch divides by va + vb + vc = 0.  The seed generator keeps
// this behaviour (the reference's); mesh_dist.cu replaces a non-finite result by its own fallback (face_dist2 there).
static __device__ V3 point_tri(V3 a, V3 b, V3 c, V3 p) {
  const V3 ab = vsub(b, a), ac = vsub(c, a), bc = vsub(c, b);
  const double snom = vdot(vsub(p, a), ab), sdenom = vdot(vsub(p, b), vsub(a, b));
  const double tnom = vdot(vsub(p, a), ac), tdenom = vdot(vsub(p, c), vsub(a, c));
  if (snom <= 0.0 && tnom <= 0.0) return a;
  const double unom = vdot(vsub(p, b), bc), udenom = vdot(vsub(p, c), vsub(b, c));
  if (sdenom <= 0.0 && unom <= 0.0) return b;
  if (tdenom <= 0.0 && udenom <= 0.0) return c;
  const V3 n = vcross(vsub(b, a), vsub(c, a));
  const double vc = vdot(n, vcross(vsub(a, p), vsub(b, p)));
  if (vc <= 0.0 && snom >= 0.0 && sdenom >= 0.0) return vadd(a, vdiv(vmul(ab, snom), snom + sdenom));
  const double va = vdot(n, vcross(vsub(b, p), vsub(c, p)));
  if (va <= 0.0 && unom >= 0.0 && udenom >= 0.0) return vadd(b, vdiv(vmul(bc, unom), unom + udenom));
  const double vb = vdot(n, vcross(vsub(c, p), vsub(a, p)));
  if (vb <= 0.0 && tnom >= 0.0 && tdenom >= 0.0) return vadd(a, vdiv(vmul(ac, tnom), tnom + tdenom));
  const double u = va / (va + vb + vc);
  const double v = vb / (va + vb + vc);
  const double w = 1.0 - u - v;
  return vadd(vadd(vmul(a, u), vmul(b, v)), vmul(c, w));
}

}  // namespace sapcu

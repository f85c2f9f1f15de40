// Host side of the triangle-mesh ground (dyros_sim_set_triangle_mesh; MeshGround in internal.h): the kept triangles and
// their bucket grid, built once when the mesh is registered. Shared with the test-only host emulation.
#pragma once
#include <string.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "internal.h"

namespace dyros {

struct MeshGrid {
  std::vector<float4> tri;  // (T, 3) MeshGround.tri
  std::vector<int4> cell;   // MeshGround.cell
  std::vector<int> list;    // MeshGround.list
  MeshGround g{};           // grid geometry, margin, ztop and zmax (pointers unset)
  long long dropped = 0;    // zero-area triangles
  long long kept = 0;
};

#define MREQ(cond, ...)                                     \
  do {                                                      \
    if (!(cond)) {                                          \
      char buf_[512];                                       \
      snprintf(buf_, sizeof buf_, __VA_ARGS__);             \
      return std::string(buf_);                             \
    }                                                       \
  } while (0)

// Validates the mesh, drops its zero-area triangles and builds the grid for query margin M = margin; "" or the error.
inline std::string build_mesh_grid(const DyrosTriangleMesh* mesh, double margin, MeshGrid& out) {
  MREQ(mesh->vertices && mesh->triangles, "vertices or triangles is NULL");
  MREQ(mesh->num_vertices >= 3 && mesh->num_triangles >= 1 && mesh->num_triangles < (1ll << 30),
       "need >= 3 vertices and 1 .. 2^30 - 1 triangles (got %lld, %lld)", (long long)mesh->num_vertices,
       (long long)mesh->num_triangles);
  MREQ(std::isfinite(mesh->origin[0]) && std::isfinite(mesh->origin[1]) && std::isfinite(mesh->origin[2]),
       "origin must be finite");
  MREQ(std::isfinite(mesh->dynamic_friction) && mesh->dynamic_friction >= 0, "dynamic_friction must be finite and >= 0");
  const int64_t nv = mesh->num_vertices, nt = mesh->num_triangles;
  for (int64_t i = 0; i < 3 * nv; ++i) MREQ(std::isfinite(mesh->vertices[i]), "vertex %lld is not finite", (long long)(i / 3));
  for (int64_t i = 0; i < 3 * nt; ++i)
    MREQ(mesh->triangles[i] < (uint64_t)nv, "triangle %lld has vertex index %u >= %lld", (long long)(i / 3),
         mesh->triangles[i], (long long)nv);
  // kept triangles: a, b - a, c - a in world coordinates, face normal in the w components
  std::vector<float4>& tri = out.tri;
  tri.clear();
  tri.reserve((size_t)nt * 3);
  std::vector<double> bx;  // x-y bounds and top of each kept triangle
  bx.reserve((size_t)nt * 5);
  std::vector<char> down;
  long long dropped = 0;
  double xmin = 1e300, ymin = 1e300, xmax = -1e300, ymax = -1e300, ztop = -1e300;
  bool any_down = false;
  for (int64_t t = 0; t < nt; ++t) {
    double P[3][3];
    for (int k = 0; k < 3; ++k)
      for (int c = 0; c < 3; ++c) P[k][c] = (double)mesh->vertices[3 * (size_t)mesh->triangles[3 * t + k] + c] + mesh->origin[c];
    const double e1[3] = {P[1][0] - P[0][0], P[1][1] - P[0][1], P[1][2] - P[0][2]};
    const double e2[3] = {P[2][0] - P[0][0], P[2][1] - P[0][1], P[2][2] - P[0][2]};
    const double n[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
    const double len = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    if (!(len > 1e-12)) {  // zero area (|cross| = twice the area, m^2)
      ++dropped;
      continue;
    }
    tri.push_back(make_float4((float)P[0][0], (float)P[0][1], (float)P[0][2], (float)(n[0] / len)));
    tri.push_back(make_float4((float)e1[0], (float)e1[1], (float)e1[2], (float)(n[1] / len)));
    tri.push_back(make_float4((float)e2[0], (float)e2[1], (float)e2[2], (float)(n[2] / len)));
    const double lo_x = std::min({P[0][0], P[1][0], P[2][0]}), hi_x = std::max({P[0][0], P[1][0], P[2][0]});
    const double lo_y = std::min({P[0][1], P[1][1], P[2][1]}), hi_y = std::max({P[0][1], P[1][1], P[2][1]});
    const double top = std::max({P[0][2], P[1][2], P[2][2]});
    bx.insert(bx.end(), {lo_x, lo_y, hi_x, hi_y, top});
    const bool dn = n[2] / len < 1e-6;  // (a wall or a face turned down: see MeshGround.cell)
    down.push_back(dn ? 1 : 0);
    any_down |= dn;
    xmin = std::min(xmin, lo_x); ymin = std::min(ymin, lo_y); xmax = std::max(xmax, hi_x); ymax = std::max(ymax, hi_y);
    ztop = std::max(ztop, top);
  }
  const int64_t nk = (int64_t)down.size();
  MREQ(nk > 0, "every one of the %lld triangles has zero area", (long long)nt);
  const double M = margin, B = kMeshBucket;
  const double x0 = xmin - M, y0 = ymin - M;
  const long long gx = (long long)std::floor((xmax + M - x0) / B) + 1, gy = (long long)std::floor((ymax + M - y0) / B) + 1;
  MREQ(gx * gy <= kMeshMaxCells, "the mesh spans %lld x %lld buckets of %g m, more than "
          "the grid's %lld", gx, gy, B, kMeshMaxCells);
  auto range = [&](int64_t t, long long& i0, long long& i1, long long& j0, long long& j1) {
    const double* b = &bx[5 * t];
    i0 = std::max(0ll, (long long)std::floor((b[0] - M - x0) / B));
    j0 = std::max(0ll, (long long)std::floor((b[1] - M - y0) / B));
    i1 = std::min(gx - 1, (long long)std::floor((b[2] + M - x0) / B));
    j1 = std::min(gy - 1, (long long)std::floor((b[3] + M - y0) / B));
  };
  std::vector<int4>& cell = out.cell;
  cell.assign((size_t)(gx * gy), make_int4(0, 0, 0, 0));
  std::vector<float> top((size_t)(gx * gy), -INFINITY), bound((size_t)(gx * gy), -INFINITY);
  long long entries = 0;
  for (int64_t t = 0; t < nk; ++t) {
    long long i0, i1, j0, j1;
    range(t, i0, i1, j0, j1);
    for (long long j = j0; j <= j1; ++j)
      for (long long i = i0; i <= i1; ++i) {
        const size_t c = (size_t)(j * gx + i);
        MREQ(cell[c].y < kMeshBucketCap, "more than %d triangles lie within the query "
                "margin of bucket (%lld, %lld) (%g m wide)", kMeshBucketCap, i, j, B);
        ++cell[c].y;
        // (rounded up: the cull stays conservative)
        top[c] = std::max(top[c], std::nextafter((float)bx[5 * t + 4], INFINITY));
        bound[c] = down[t] ? INFINITY : std::max(bound[c], top[c]);
      }
    entries += (i1 - i0 + 1) * (j1 - j0 + 1);
  }
  MREQ(entries < (1ll << 31), "the grid would hold %lld entries (limit 2^31)", entries);
  long long off = 0;
  for (size_t c = 0; c < cell.size(); ++c) {
    cell[c].x = (int)off;
    off += cell[c].y;
    memcpy(&cell[c].z, &bound[c], 4);
    memcpy(&cell[c].w, &top[c], 4);
    cell[c].y = 0;  // (refilled below)
  }
  std::vector<int>& list = out.list;
  list.assign((size_t)entries, 0);
  for (int64_t t = 0; t < nk; ++t) {
    long long i0, i1, j0, j1;
    range(t, i0, i1, j0, j1);
    for (long long j = j0; j <= j1; ++j)
      for (long long i = i0; i <= i1; ++i) {
        int4& c = cell[(size_t)(j * gx + i)];
        list[(size_t)c.x + c.y++] = (int)t;
      }
  }
  MeshGround& g = out.g;
  g = MeshGround{};
  g.gx = (int)gx;
  g.gy = (int)gy;
  g.x0 = (float)x0;
  g.y0 = (float)y0;
  g.inv_b = (float)(1 / B);
  g.margin = (float)M;
  g.ztop = std::nextafter((float)ztop, INFINITY);
  g.zmax = any_down ? INFINITY : g.ztop;
  out.dropped = dropped;
  out.kept = nk;
  return "";
}
#undef MREQ

}  // namespace dyros

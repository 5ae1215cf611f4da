// Internal declarations of the lattice isosurface (isosurface.cu): the handle behind the fr_isosurface_* entry points
// and the device stages that fr_isosurface_extract (solver.cu) strings together around the model's evaluations.
#pragma once
#include <functional>
#include <memory>
#include <vector>

#include "fmm.h"

namespace fb {

constexpr uint64_t kIsoMaxNodes = 1ull << 28;  // about 100 B of device memory per node with the binning buffers

// lattice of resolution n per axis over [lo, hi]: node idx is idx * step + lo, the last node exactly hi (np.linspace)
struct IsoLattice {
  uint64_t n[3] = {0, 0, 0};
  double lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0}, step[3] = {0, 0, 0};
  __host__ __device__ uint64_t nodes() const { return n[0] * n[1] * n[2]; }
  __host__ __device__ uint64_t cubes() const { return (n[0] - 1) * (n[1] - 1) * (n[2] - 1); }
};
// FB_ERR_INVALID_ARGUMENT unless lo < hi (finite) and n >= 2 on every axis and the node count is at most kIsoMaxNodes
IsoLattice iso_lattice(const double *extents, const uint64_t *resolution);

constexpr int kIsoOpen = -1;  // IsoSurface::side of an open isosurface; 0 = the solid {f < iso}, 1 = {f >= iso}

struct IsoSurface {
  double iso = 0;
  int side = kIsoOpen;
  uint64_t nv = 0, nf = 0;           // isosurface vertices and faces
  uint64_t cv = 0, cf = 0;           // solids: cap nodes and cap faces, after the isosurface's in verts and faces
  DBuf<double> verts, normals;       // (nv + cv) x 3 row-major
  DBuf<long long> faces;             // (nf + cf) x 3 row-major
  DBuf<unsigned long long> edge;     // edge id of every isosurface vertex, 7 p(a) + mask - 1
  DBuf<unsigned long long> cap_node; // lattice node of every cap vertex
  bool has_normals = false;
  uint64_t evaluations = 0, max_iterations = 0;  // refinement: trial points evaluated, iterations of the slowest vertex
  double volume = 0, area = 0;       // solids: enclosed volume, area of the isosurface faces
};

// regula falsi state of one vertex: bracket [ta, tb] on its edge a -> b with f - iso at both ends, next trial t
struct IsoRefine {
  double ta, tb, fa, fb, t;
  int last;   // side replaced by the previous step: 0 = a, 1 = b, -1 = none
  int iters;
};

// device scratch of one extraction call, reused across its isovalues
struct IsoScratch {
  DBuf<uint8_t> mask, ccount;               // per node: crossing edges (bits 0-6) and class (bit 7); per cube: triangles
  DBuf<unsigned long long> voff, foff, bad;  // vertex / face offsets (scans), first non-finite value
  DBuf<unsigned char> cub;
  DBuf<unsigned long long> act[2];          // refinement: active vertices
  DBuf<uint8_t> keep;
  DBuf<int> n_sel;
  DBuf<IsoRefine> state;
  DBuf<double> pts, vals;
  DBuf<unsigned long long> coff, soff;      // solids: cap node offsets per boundary node, cap face offsets per square
  DBuf<uint8_t> scount;                     // solids: cap faces per box-face square
  DBuf<double> sums;                        // solids: volume and area sums
};

// node coordinates, n x 3 row-major, node p = i + nx * (j + ny * k)
void iso_lattice_points(const IsoLattice &L, double *d_xyz, cudaStream_t s);
// index of the first non-finite value of d_v[p * stride], or the node count when all are finite; blocks
uint64_t iso_first_nonfinite(const double *d_v, size_t stride, uint64_t n, IsoScratch &w, cudaStream_t s);
// vertices and faces of the level set `out.iso` of the lattice values d_v[p * stride], and for out.side >= 0 the cap
// nodes and faces that close it into a solid; blocks once for the counts
void iso_extract(const double *d_v, size_t stride, const IsoLattice &L, IsoScratch &w, IsoSurface &out, cudaStream_t s);
// evaluates the interpolant at m points (m x 3 row-major, device) into vals (m x n_cols row-major, device), on s
using IsoEval = std::function<void(const double *pts, size_t m, double *vals)>;
// Illinois regula falsi on every vertex's edge, the lattice values as the first bracket
void iso_refine(const double *d_v, size_t stride, const IsoLattice &L, int n_cols, int col, const IsoEval &eval,
                IsoScratch &w, IsoSurface &surf, cudaStream_t s);
// normals[v] = gradient of column col at vertex v (d_grads: nv x (n_cols * 3) row-major), normalised; for solids negated
// on side 1, and on the cap nodes the normalised sum of the outward normals of the box faces they lie on
void iso_normals(const double *d_grads, int n_cols, int col, const IsoLattice &L, IsoSurface &surf, cudaStream_t s);
// solids: volume and isosurface area from the final vertex positions, by fixed-order reductions; blocks
void iso_measure(const IsoLattice &L, IsoScratch &w, IsoSurface &surf, cudaStream_t s);

}  // namespace fb

struct fr_isosurface {
  int device = 0;
  std::vector<std::unique_ptr<fb::IsoSurface>> surf;
  double ms[4] = {0, 0, 0, 0};  // lattice evaluation (tree included), extraction, refinement, normals
};

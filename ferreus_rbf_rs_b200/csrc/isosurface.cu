// Isosurfaces of lattice values (fr_lattice_isosurface, and the extraction stages of fr_isosurface_extract in
// solver.cu): lattice generator, crossing masks and their scan, vertex emission, per-cube triangle counts, their scan
// and triangle emission, the regula falsi update of the refinement with its compaction, and the normals.
// The mesh is fixed by a specification that tests/isosurface_oracle.py restates (DESIGN.md, "Isosurfaces"):
//  - node p = i + nx (j + ny k) is below when v < iso (a tie is not below);
//  - every cube is split into the 6 Kuhn tetrahedra (c, c + e[pi0], c + e[pi0] + e[pi1], c + (1,1,1)), pi in
//    lexicographic order, so every edge runs from a node a to a + s, s a nonzero 0/1 vector of mask sx + 2 sy + 4 sz;
//  - one vertex per crossing edge, numbered by its edge id 7 p(a) + mask - 1: the node's base (a scan of the
//    popcounts of the 7-bit crossing masks) plus the popcount of the mask's lower bits;
//  - triangles in the order (cube, pi, triangle), oriented by kSwap from the below side to the other side.
// Solids (fr_lattice_solid, fr_isosurface_extract_solid) close that mesh at the lattice box with caps built from the
// boundary nodes of the solid's side and the existing rim vertices (tests/solid_oracle.py, DESIGN.md "Solids"), and
// reduce the volume and the isosurface area from the final vertices.
#include "isosurface.h"

#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include <chrono>
#include <cmath>

namespace fb {
namespace {

inline unsigned nblocks(uint64_t n, int bs) { return (unsigned)((n + bs - 1) / bs); }

// bit 2 * mask + tri of kSwap[pi]: exchange the triangle's last two vertices.  Decided once on the edge midpoints of
// the unit cube (tests/isosurface_oracle.py, swap_table), not per triangle from coordinates, so triangles made
// degenerate by a value equal to iso are oriented like their neighbours.  120 entries are used.
__constant__ uint32_t kSwap[6] = {0x10710c10u, 0x070c71c4u, 0x070c71c4u, 0x10710c10u, 0x10710c10u, 0x070c71c4u};
// first two axes of the permutations 012, 021, 102, 120, 201, 210
__constant__ uint8_t kPi[6][2] = {{0, 1}, {0, 2}, {1, 0}, {1, 2}, {2, 0}, {2, 1}};

__host__ __device__ __forceinline__ unsigned popc(unsigned x) {
#ifdef __CUDA_ARCH__
  return __popc(x);
#else
  return (unsigned)__builtin_popcount(x);
#endif
}

// node idx on axis d, rounded as np.linspace: idx * step + lo, the last node exactly hi
__device__ __forceinline__ double coord(const IsoLattice &L, int d, uint64_t idx) {
  return idx == L.n[d] - 1 ? L.hi[d] : __dadd_rn(__dmul_rn((double)idx, L.step[d]), L.lo[d]);
}

__device__ __forceinline__ uint64_t node_offset(const IsoLattice &L, unsigned s) {  // a + s - a for mask s
  return (s & 1) + L.n[0] * (((s >> 1) & 1) + L.n[1] * (s >> 2));
}

// position on the edge a -> a + s at parameter t, every operation rounded on its own
__device__ __forceinline__ void edge_point(const IsoLattice &L, uint64_t a, unsigned s, double t, double *out) {
  const uint64_t idx[3] = {a % L.n[0], (a / L.n[0]) % L.n[1], a / (L.n[0] * L.n[1])};
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const double xa = coord(L, d, idx[d]), xb = coord(L, d, idx[d] + ((s >> d) & 1));
    out[d] = __dadd_rn(xa, __dmul_rn(t, __dsub_rn(xb, xa)));
  }
}

__global__ void k_iso_lattice(IsoLattice L, double *__restrict__ xyz) {
  const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (p >= L.nodes()) return;
  const uint64_t i = p % L.n[0], r = p / L.n[0];
  xyz[3 * p] = coord(L, 0, i);
  xyz[3 * p + 1] = coord(L, 1, r % L.n[1]);
  xyz[3 * p + 2] = coord(L, 2, r / L.n[1]);
}

__global__ void k_iso_nonfinite(const double *__restrict__ v, size_t stride, uint64_t n, unsigned long long *first) {
  const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (p < n && !isfinite(v[p * stride])) atomicMin(first, (unsigned long long)p);
}

// per node: bit s - 1 = the edge a -> a + s crosses (s = 1..7, the other end inside the lattice), bit 7 = below
__global__ void k_iso_masks(const double *__restrict__ v, size_t stride, IsoLattice L, double iso,
                            uint8_t *__restrict__ mask) {
  const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (p >= L.nodes()) return;
  const uint64_t i = p % L.n[0], r = p / L.n[0], j = r % L.n[1], k = r / L.n[1];
  const bool below = v[p * stride] < iso;
  unsigned m = below ? 0x80u : 0u;
#pragma unroll
  for (unsigned s = 1; s < 8; ++s) {
    if (i + (s & 1) >= L.n[0] || j + ((s >> 1) & 1) >= L.n[1] || k + (s >> 2) >= L.n[2]) continue;
    if ((v[(p + node_offset(L, s)) * stride] < iso) != below) m |= 1u << (s - 1);
  }
  mask[p] = (uint8_t)m;
}

struct NodeVertices {  // vertices owned by node p; 0 past the end (the scan's n + 1st element is the total)
  const uint8_t *mask;
  uint64_t n;
  __host__ __device__ unsigned long long operator()(uint64_t p) const { return p < n ? popc(mask[p] & 0x7fu) : 0; }
};

struct CubeFaces {  // also the cap faces per box-face square
  const uint8_t *count;
  uint64_t n;
  __host__ __device__ unsigned long long operator()(uint64_t c) const { return c < n ? count[c] : 0; }
};

// exclusive scan of f(0 .. n) into out[0 .. n]: out[n] is the total
template <class F>
void scan_counts(F f, uint64_t n, unsigned long long *out, IsoScratch &w, cudaStream_t s) {
  auto in = thrust::make_transform_iterator(thrust::counting_iterator<uint64_t>(0), f);
  size_t bytes = 0;
  FB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, (int)(n + 1), s));
  w.cub.reserve(bytes);
  FB_CUDA(cub::DeviceScan::ExclusiveSum(w.cub.p, bytes, in, out, (int)(n + 1), s));
  g_launches.fetch_add(1);
}

__global__ void k_iso_vertices(const double *__restrict__ v, size_t stride, IsoLattice L, double iso,
                               const uint8_t *__restrict__ mask, const unsigned long long *__restrict__ voff,
                               double *__restrict__ verts, unsigned long long *__restrict__ edge) {
  const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (p >= L.nodes()) return;
  const unsigned m = mask[p] & 0x7fu;
  if (!m) return;
  const double va = v[p * stride];
  unsigned long long o = voff[p];
  for (unsigned s = 1; s < 8; ++s) {
    if (!((m >> (s - 1)) & 1)) continue;
    const double vb = v[(p + node_offset(L, s)) * stride];
    const double t = __ddiv_rn(__dsub_rn(iso, va), __dsub_rn(vb, va));
    edge_point(L, p, s, t, verts + 3 * o);
    edge[o] = 7 * p + (s - 1);
    ++o;
  }
}

// classes of a cube's 8 corners (bit ox + 2 oy + 4 oz = corner is below) and the node of its minimum corner
__device__ __forceinline__ unsigned cube_classes(const uint8_t *__restrict__ mask, const IsoLattice &L, uint64_t c,
                                                 uint64_t &base) {
  const uint64_t cx = L.n[0] - 1, cy = L.n[1] - 1;
  const uint64_t ci = c % cx, r = c / cx;
  base = ci + L.n[0] * (r % cy + L.n[1] * (r / cy));
  unsigned cls = 0;
#pragma unroll
  for (unsigned o = 0; o < 8; ++o) cls |= (unsigned)(mask[base + node_offset(L, o)] >> 7) << o;
  return cls;
}

// corner of chain position q (0..3) of tetrahedron pi, as a corner bit set
__device__ __forceinline__ unsigned chain_corner(int pi, int q) {
  const unsigned c1 = 1u << kPi[pi][0];
  return q == 0 ? 0u : q == 1 ? c1 : q == 2 ? (c1 | 1u << kPi[pi][1]) : 7u;
}

// below mask of tetrahedron pi: bit q = chain position q is below
__device__ __forceinline__ unsigned tet_mask(unsigned cls, int pi) {
  unsigned m = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) m |= ((cls >> chain_corner(pi, q)) & 1u) << q;
  return m;
}

__device__ __forceinline__ unsigned tet_triangles(unsigned m) {
  const unsigned nb = popc(m);
  return nb == 2 ? 2u : (nb == 1 || nb == 3) ? 1u : 0u;
}

__global__ void k_iso_cube_counts(const uint8_t *__restrict__ mask, IsoLattice L, uint8_t *__restrict__ count) {
  const uint64_t c = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (c >= L.cubes()) return;
  uint64_t base;
  const unsigned cls = cube_classes(mask, L, c, base);
  unsigned n = 0;
  if (cls != 0 && cls != 0xffu)
#pragma unroll
    for (int pi = 0; pi < 6; ++pi) n += tet_triangles(tet_mask(cls, pi));
  count[c] = (uint8_t)n;
}

// vertex of the edge between chain positions u < w of tetrahedron pi
__device__ __forceinline__ long long tet_vertex(const uint8_t *__restrict__ mask,
                                                const unsigned long long *__restrict__ voff, const IsoLattice &L,
                                                uint64_t base, int pi, unsigned u, unsigned w) {
  const unsigned cu = chain_corner(pi, u), s = chain_corner(pi, w) & ~cu;
  const uint64_t a = base + node_offset(L, cu);
  return (long long)(voff[a] + popc(mask[a] & ((1u << (s - 1)) - 1u)));
}

// triangles of one tetrahedron as chain-position pairs, 2 bits each: (u0 w0 u1 w1 u2 w2) per triangle
__device__ __forceinline__ void tet_pairs(unsigned m, unsigned &t0, unsigned &t1) {
  auto pair3 = [](unsigned a, unsigned b, unsigned c, unsigned d, unsigned e, unsigned f) {
    return a | b << 2 | c << 4 | d << 6 | e << 8 | f << 10;
  };
  const unsigned nb = popc(m);
  if (nb == 2) {  // a < b below, c < d not below: (a,c) (a,d) (b,d) and (a,c) (b,d) (b,c)
    const unsigned a = __ffs(m) - 1, b = 31 - __clz(m), na = ~m & 15u;
    const unsigned c = __ffs(na) - 1, d = 31 - __clz(na);
    t0 = pair3(a, c, a, d, b, d);
    t1 = pair3(a, c, b, d, b, c);
    return;
  }
  // the lone corner q against the others r1 < r2 < r3
  const unsigned lone = nb == 1 ? m : ~m & 15u, q = __ffs(lone) - 1;
  unsigned rest = 15u & ~lone;
  const unsigned r1 = __ffs(rest) - 1;
  rest &= rest - 1;
  const unsigned r2 = __ffs(rest) - 1, r3 = 31 - __clz(rest);
  t0 = pair3(q, r1, q, r2, q, r3);
  t1 = 0;
}

// flip (the solid above the level set) exchanges every triangle's last two vertices, so that it faces out of the solid
__global__ void k_iso_triangles(const uint8_t *__restrict__ mask, IsoLattice L,
                                const unsigned long long *__restrict__ voff, const unsigned long long *__restrict__ foff,
                                bool flip, long long *__restrict__ faces) {
  const uint64_t c = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (c >= L.cubes()) return;
  uint64_t base;
  const unsigned cls = cube_classes(mask, L, c, base);
  if (cls == 0 || cls == 0xffu) return;
  unsigned long long f = foff[c];
  for (int pi = 0; pi < 6; ++pi) {
    const unsigned m = tet_mask(cls, pi), nt = tet_triangles(m);
    if (!nt) continue;
    unsigned tp[2];
    tet_pairs(m, tp[0], tp[1]);
    for (unsigned t = 0; t < nt; ++t) {
      long long vid[3];
#pragma unroll
      for (int e = 0; e < 3; ++e) {
        const unsigned x = (tp[t] >> (4 * e)) & 3u, y = (tp[t] >> (4 * e + 2)) & 3u;
        vid[e] = tet_vertex(mask, voff, L, base, pi, x < y ? x : y, x < y ? y : x);
      }
      const bool swap = (bool)((kSwap[pi] >> (2 * m + t)) & 1u) != flip;
      faces[3 * f] = vid[0];
      faces[3 * f + 1] = swap ? vid[2] : vid[1];
      faces[3 * f + 2] = swap ? vid[1] : vid[2];
      ++f;
    }
  }
}

// ------------------------------------------------------------------------------------------- solids
// The caps close the isosurface at the lattice box.  On box face f (0-5: x lo, x hi, y lo, y hi, z lo, z hi; in-plane
// axes u < v) square (au, av) has index au + (nu - 1) av and the triangles T0 = (a, a + e_u, a + e_u + e_v) and
// T1 = (a, a + e_v, a + e_u + e_v), the boundary faces of the Kuhn tetrahedra, so every triangle edge is a lattice edge
// with its vertex already numbered.  A triangle is clipped to the solid's side: one inside corner q against r1 < r2
// gives (q, e(q,r1), e(q,r2)); two inside corners q1 < q2 against r give (q1, q2, e(q2,r)) and (q1, e(q2,r), e(q1,r));
// three give the triangle.  Cap vertices are the boundary nodes of the solid's side in ascending node index.

// bit 2 (8 tri + inside mask) + sub-triangle of kCapSwap[box face]: exchange the sub-triangle's last two vertices so
// that (B-A) x (C-A) points out of the box.  Decided once on the unit square with the crossing points at the edge
// midpoints (tests/solid_oracle.py, cap_swap_table), like kSwap.
__constant__ uint32_t kCapSwap[6] = {0x0c1071c4u, 0x71c40c10u, 0x71c40c10u, 0x0c1071c4u, 0x0c1071c4u, 0x71c40c10u};

// the class bit of a node's mask against the solid's side: side 0 holds the below nodes, side 1 the others
__host__ __device__ __forceinline__ unsigned inside(uint8_t m, unsigned side) { return (unsigned)(m >> 7) ^ side; }

__host__ __device__ __forceinline__ uint64_t boundary_count(const IsoLattice &L) {
  return L.nodes() - (L.n[0] - 2) * (L.n[1] - 2) * (L.n[2] - 2);
}

// Boundary nodes in ascending node index: the k = 0 layer, then per inner layer its j = 0 row, the i = 0 and
// i = nx - 1 nodes of its inner rows and its j = ny - 1 row (2 nx + 2 (ny - 2) nodes), then the k = nz - 1 layer.
__host__ __device__ __forceinline__ uint64_t boundary_node(const IsoLattice &L, uint64_t b) {
  const uint64_t nx = L.n[0], ny = L.n[1], layer = nx * ny, ring = 2 * nx + 2 * (ny - 2), inner = (L.n[2] - 2) * ring;
  if (b < layer) return b;
  b -= layer;
  if (b >= inner) return L.nodes() - layer + (b - inner);
  const uint64_t k = 1 + b / ring, r = b % ring;
  uint64_t i, j;
  if (r < nx) {
    i = r;
    j = 0;
  } else if (r >= ring - nx) {
    i = r - (ring - nx);
    j = ny - 1;
  } else {
    j = 1 + (r - nx) / 2;
    i = ((r - nx) & 1) ? nx - 1 : 0;
  }
  return i + nx * (j + ny * k);
}

// inverse of boundary_node for a node p on the boundary
__device__ __forceinline__ uint64_t boundary_rank(const IsoLattice &L, uint64_t p) {
  const uint64_t nx = L.n[0], ny = L.n[1], layer = nx * ny, ring = 2 * nx + 2 * (ny - 2);
  const uint64_t i = p % nx, j = (p / nx) % ny, k = p / layer;
  if (k == 0) return p;
  if (k == L.n[2] - 1) return layer + (L.n[2] - 2) * ring + (p - k * layer);
  const uint64_t b = layer + (k - 1) * ring;
  if (j == 0) return b + i;
  if (j == ny - 1) return b + ring - nx + i;
  return b + nx + 2 * (j - 1) + (i != 0);
}

struct CapNodes {  // 1 for a boundary node of the solid's side; 0 past the end
  const uint8_t *mask;
  IsoLattice L;
  unsigned side;
  uint64_t n;
  __host__ __device__ unsigned long long operator()(uint64_t b) const {
    return b < n ? inside(mask[boundary_node(L, b)], side) : 0;
  }
};

// first square of every box face (start[6] = all squares)
struct CapSquares {
  uint64_t start[7];
};

CapSquares cap_squares(const IsoLattice &L) {
  CapSquares S;
  S.start[0] = 0;
  for (int f = 0; f < 6; ++f) {
    const int w = f / 2, u = w == 0 ? 1 : 0, v = w == 2 ? 1 : 2;
    S.start[f + 1] = S.start[f] + (L.n[u] - 1) * (L.n[v] - 1);
  }
  return S;
}

__device__ __forceinline__ uint64_t axis_n(const IsoLattice &L, int d) { return d == 0 ? L.n[0] : d == 1 ? L.n[1] : L.n[2]; }
__device__ __forceinline__ uint64_t axis_stride(const IsoLattice &L, int d) {
  return d == 0 ? 1 : d == 1 ? L.n[0] : L.n[0] * L.n[1];
}

// square g of all box faces: its box face, the node of its minimum corner and the edge masks of e_u and e_v
// (selects rather than indexed arrays keep the kernels free of a stack frame)
__device__ __forceinline__ int cap_square(const IsoLattice &L, const CapSquares &S, uint64_t g, uint64_t &a,
                                          unsigned &su, unsigned &sv) {
  int f = 0;
  uint64_t first = 0;
#pragma unroll
  for (int k = 1; k < 6; ++k)
    if (g >= S.start[k]) {
      f = k;
      first = S.start[k];
    }
  const uint64_t q = g - first;
  const int w = f / 2, u = w == 0 ? 1 : 0, v = w == 2 ? 1 : 2;
  const uint64_t nu1 = axis_n(L, u) - 1;
  a = (q % nu1) * axis_stride(L, u) + (q / nu1) * axis_stride(L, v) +
      ((f & 1) ? (axis_n(L, w) - 1) * axis_stride(L, w) : 0);
  su = 1u << u;
  sv = 1u << v;
  return f;
}

// corner q of triangle t of a square, as an edge mask from the square's minimum corner: (0, e_u or e_v, e_u + e_v)
__device__ __forceinline__ unsigned cap_corner(unsigned su, unsigned sv, int t, unsigned q) {
  return q == 0 ? 0u : q == 1 ? (t ? sv : su) : (su | sv);
}

// inside mask of triangle t of a square: bit q = corner q is inside
__device__ __forceinline__ unsigned cap_triangle(const uint8_t *__restrict__ mask, const IsoLattice &L, uint64_t a,
                                                 unsigned su, unsigned sv, int t, unsigned side) {
  unsigned m = 0;
#pragma unroll
  for (unsigned q = 0; q < 3; ++q) m |= inside(mask[a + node_offset(L, cap_corner(su, sv, t, q))], side) << q;
  return m;
}

__device__ __forceinline__ unsigned cap_subtriangles(unsigned m) {
  const unsigned n = popc(m);
  return n == 2 ? 2u : n ? 1u : 0u;
}

__global__ void k_iso_cap_counts(const uint8_t *__restrict__ mask, IsoLattice L, CapSquares S, unsigned side,
                                 uint8_t *__restrict__ count) {
  const uint64_t g = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (g >= S.start[6]) return;
  uint64_t a;
  unsigned su, sv;
  cap_square(L, S, g, a, su, sv);
  count[g] = (uint8_t)(cap_subtriangles(cap_triangle(mask, L, a, su, sv, 0, side)) +
                       cap_subtriangles(cap_triangle(mask, L, a, su, sv, 1, side)));
}

__global__ void k_iso_cap_nodes(const uint8_t *__restrict__ mask, IsoLattice L, unsigned side,
                                const unsigned long long *__restrict__ coff, uint64_t nv, double *__restrict__ verts,
                                unsigned long long *__restrict__ cap_node) {
  const uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (b >= boundary_count(L)) return;
  const uint64_t p = boundary_node(L, b);
  if (!inside(mask[p], side)) return;
  const unsigned long long o = coff[b];
  const uint64_t idx[3] = {p % L.n[0], (p / L.n[0]) % L.n[1], p / (L.n[0] * L.n[1])};
#pragma unroll
  for (int d = 0; d < 3; ++d) verts[3 * (nv + o) + d] = coord(L, d, idx[d]);
  cap_node[o] = p;
}

__global__ void k_iso_cap_faces(const uint8_t *__restrict__ mask, IsoLattice L, CapSquares S, unsigned side,
                                const unsigned long long *__restrict__ voff, const unsigned long long *__restrict__ coff,
                                const unsigned long long *__restrict__ soff, uint64_t nv, uint64_t nf,
                                long long *__restrict__ faces) {
  const uint64_t g = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (g >= S.start[6]) return;
  uint64_t a;
  unsigned su, sv;
  const int f = cap_square(L, S, g, a, su, sv);
  unsigned long long o = nf + soff[g];
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const unsigned m = cap_triangle(mask, L, a, su, sv, t, side);
    if (!m) continue;
    auto node = [&](unsigned q) {
      return (long long)(nv + coff[boundary_rank(L, a + node_offset(L, cap_corner(su, sv, t, q)))]);
    };
    auto rim = [&](unsigned q, unsigned r) {  // vertex of the edge between corners q and r, numbered as tet_vertex
      const unsigned cl = cap_corner(su, sv, t, q < r ? q : r), s = cap_corner(su, sv, t, q < r ? r : q) & ~cl;
      const uint64_t x = a + node_offset(L, cl);
      return (long long)(voff[x] + popc(mask[x] & ((1u << (s - 1)) - 1u)));
    };
    long long v0[3], v1[3];
    const unsigned n = popc(m);
    if (n == 3) {
      v0[0] = node(0);
      v0[1] = node(1);
      v0[2] = node(2);
    } else {
      const unsigned lone = n == 1 ? m : ~m & 7u, q = __ffs(lone) - 1, r1 = __ffs(7u & ~lone) - 1,
                     r2 = 31 - __clz(7u & ~lone);
      if (n == 1) {
        v0[0] = node(q);
        v0[1] = rim(q, r1);
        v0[2] = rim(q, r2);
      } else {  // inside r1 < r2, outside q
        v0[0] = node(r1);
        v0[1] = node(r2);
        v0[2] = rim(r2, q);
        v1[0] = v0[0];
        v1[1] = v0[2];
        v1[2] = rim(r1, q);
      }
    }
#pragma unroll
    for (unsigned k = 0; k < 2; ++k) {
      if (k == 1 && n != 2) break;
      const long long *vid = k ? v1 : v0;
      const bool swap = (kCapSwap[f] >> (2 * (8 * t + m) + k)) & 1u;
      faces[3 * o] = vid[0];
      faces[3 * o + 1] = swap ? vid[2] : vid[1];
      faces[3 * o + 2] = swap ? vid[1] : vid[2];
      ++o;
    }
  }
}

// 6 x the signed volume of the tetrahedron (o, A, B, C)
struct FaceVolume {
  const double *v;
  const long long *f;
  double o[3];
  __host__ __device__ double operator()(uint64_t i) const {
    double x[3][3];
    for (int e = 0; e < 3; ++e)
      for (int d = 0; d < 3; ++d) x[e][d] = v[3 * f[3 * i + e] + d] - o[d];
    return x[0][0] * (x[1][1] * x[2][2] - x[1][2] * x[2][1]) + x[0][1] * (x[1][2] * x[2][0] - x[1][0] * x[2][2]) +
           x[0][2] * (x[1][0] * x[2][1] - x[1][1] * x[2][0]);
  }
};

// 2 x the area of face i
struct FaceArea {
  const double *v;
  const long long *f;
  __host__ __device__ double operator()(uint64_t i) const {
    const double *a = v + 3 * f[3 * i], *b = v + 3 * f[3 * i + 1], *c = v + 3 * f[3 * i + 2];
    const double p[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, q[3] = {c[0] - a[0], c[1] - a[1], c[2] - a[2]};
    const double x = p[1] * q[2] - p[2] * q[1], y = p[2] * q[0] - p[0] * q[2], z = p[0] * q[1] - p[1] * q[0];
    return sqrt(x * x + y * y + z * z);
  }
};

template <class F>
void reduce_sum(F f, uint64_t n, double *out, IsoScratch &w, cudaStream_t s) {
  auto in = thrust::make_transform_iterator(thrust::counting_iterator<uint64_t>(0), f);
  size_t bytes = 0;
  FB_CUDA(cub::DeviceReduce::Sum(nullptr, bytes, in, out, (int64_t)n, s));
  w.cub.reserve(bytes);
  FB_CUDA(cub::DeviceReduce::Sum(w.cub.p, bytes, in, out, (int64_t)n, s));
  g_launches.fetch_add(1);
}

__global__ void k_iso_cap_normals(IsoLattice L, const unsigned long long *__restrict__ cap_node, uint64_t cv,
                                  double *__restrict__ nrm) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= cv) return;
  const uint64_t p = cap_node[i];
  const uint64_t idx[3] = {p % L.n[0], (p / L.n[0]) % L.n[1], p / (L.n[0] * L.n[1])};
  double n[3], len = 0.0;
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    n[d] = idx[d] == 0 ? -1.0 : idx[d] == L.n[d] - 1 ? 1.0 : 0.0;
    len += n[d] * n[d];
  }
  const double inv = 1.0 / sqrt(len);
#pragma unroll
  for (int d = 0; d < 3; ++d) nrm[3 * i + d] = n[d] * inv;
}

// ------------------------------------------------------------------------------------------- refinement
__global__ void k_iso_refine_init(const double *__restrict__ v, size_t stride, IsoLattice L, double iso,
                                  const unsigned long long *__restrict__ edge, uint64_t nv, IsoRefine *__restrict__ st,
                                  unsigned long long *__restrict__ act) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= nv) return;
  const uint64_t a = edge[i] / 7;
  const unsigned s = (unsigned)(edge[i] % 7) + 1;
  const double va = v[a * stride], vb = v[(a + node_offset(L, s)) * stride];
  IsoRefine r;
  r.ta = 0.0;
  r.tb = 1.0;
  r.fa = va - iso;
  r.fb = vb - iso;
  r.t = __ddiv_rn(__dsub_rn(iso, va), __dsub_rn(vb, va));  // the first trial is the unrefined vertex
  r.last = -1;
  r.iters = 0;
  st[i] = r;
  act[i] = i;
}

__global__ void k_iso_refine_points(IsoLattice L, const unsigned long long *__restrict__ edge,
                                    const IsoRefine *__restrict__ st, const unsigned long long *__restrict__ act,
                                    uint64_t na, double *__restrict__ pts) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= na) return;
  const unsigned long long vx = act[i];
  edge_point(L, edge[vx] / 7, (unsigned)(edge[vx] % 7) + 1, st[vx].t, pts + 3 * i);
}

// Illinois step: the trial value g replaces the bracket end of its sign class; an end kept twice in a row has its value
// halved.  Done at g == iso exactly, a bracket of at most 2^-40 of the edge, or kIsoMaxIters evaluations.
constexpr int kIsoMaxIters = 60;
__global__ void k_iso_refine_update(const double *__restrict__ vals, int n_cols, int col, double iso,
                                    const unsigned long long *__restrict__ act, uint64_t na,
                                    const double *__restrict__ pts, IsoRefine *__restrict__ st,
                                    double *__restrict__ verts, uint8_t *__restrict__ keep) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= na) return;
  const unsigned long long vx = act[i];
  IsoRefine r = st[vx];
  const double g = vals[i * n_cols + col] - iso;
  for (int d = 0; d < 3; ++d) verts[3 * vx + d] = pts[3 * i + d];
  ++r.iters;
  bool done = g == 0.0;
  if (!done) {
    if ((g < 0.0) == (r.fa < 0.0)) {
      r.ta = r.t;
      r.fa = g;
      if (r.last == 0) r.fb *= 0.5;
      r.last = 0;
    } else {
      r.tb = r.t;
      r.fb = g;
      if (r.last == 1) r.fa *= 0.5;
      r.last = 1;
    }
    done = r.tb - r.ta <= 0x1p-40 || r.iters >= kIsoMaxIters;
    if (!done) r.t = fmin(fmax(r.ta - r.fa * (r.tb - r.ta) / (r.fb - r.fa), r.ta), r.tb);
  }
  st[vx] = r;
  keep[i] = !done;
}

// negate: the solid above the level set, whose outward normal is the negated gradient
__global__ void k_iso_normals(const double *__restrict__ g, int n_cols, int col, uint64_t nv, bool negate,
                              double *__restrict__ nrm) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= nv) return;
  const double *gi = g + i * (uint64_t)(3 * n_cols) + 3 * col;
  const double x = gi[0], y = gi[1], z = gi[2];
  const double len = sqrt(x * x + y * y + z * z);
  const double inv = len > 0.0 ? (negate ? -1.0 : 1.0) / len : 0.0;
  nrm[3 * i] = x * inv;
  nrm[3 * i + 1] = y * inv;
  nrm[3 * i + 2] = z * inv;
}

}  // namespace

// ------------------------------------------------------------------------------------------------ stages
IsoLattice iso_lattice(const double *extents, const uint64_t *resolution) {
  FB_REQUIRE(extents && resolution, "extents (x0, y0, z0, x1, y1, z1) and resolution (nx, ny, nz) are required");
  IsoLattice L;
  uint64_t nodes = 1;
  for (int d = 0; d < 3; ++d) {
    const uint64_t n = resolution[d];
    FB_REQUIRE(n >= 2, "resolution must be at least 2 on every axis");
    FB_REQUIRE(n <= kIsoMaxNodes && nodes * n <= kIsoMaxNodes,
               "a lattice has at most 2^28 = " + std::to_string(kIsoMaxNodes) + " nodes");
    nodes *= n;
    const double lo = extents[d], hi = extents[3 + d];
    FB_REQUIRE(std::isfinite(lo) && std::isfinite(hi) && lo < hi && std::isfinite(hi - lo),
               "extents must be finite with lo < hi on every axis");
    L.n[d] = n;
    L.lo[d] = lo;
    L.hi[d] = hi;
    L.step[d] = (hi - lo) / (double)(n - 1);
  }
  return L;
}

void iso_lattice_points(const IsoLattice &L, double *d_xyz, cudaStream_t s) {
  FB_LAUNCH(k_iso_lattice, nblocks(L.nodes(), 256), 256, 0, s, L, d_xyz);
}

uint64_t iso_first_nonfinite(const double *d_v, size_t stride, uint64_t n, IsoScratch &w, cudaStream_t s) {
  w.bad.reserve(1);
  FB_CUDA(cudaMemsetAsync(w.bad.p, 0xFF, sizeof(unsigned long long), s));
  FB_LAUNCH(k_iso_nonfinite, nblocks(n, 256), 256, 0, s, d_v, stride, n, w.bad.p);
  unsigned long long h = 0;
  FB_CUDA(cudaMemcpyAsync(&h, w.bad.p, sizeof(h), cudaMemcpyDeviceToHost, s));
  FB_CUDA(cudaStreamSynchronize(s));
  return h == ~0ull ? n : (uint64_t)h;
}

void iso_extract(const double *d_v, size_t stride, const IsoLattice &L, IsoScratch &w, IsoSurface &out,
                 cudaStream_t s) {
  const uint64_t n = L.nodes(), nc = L.cubes();
  const bool solid = out.side != kIsoOpen;
  const unsigned side = solid ? (unsigned)out.side : 0u;
  const uint64_t nb = boundary_count(L);
  const CapSquares S = cap_squares(L);
  const uint64_t ns = S.start[6];
  w.mask.reserve(n);
  w.voff.reserve(n + 1);
  w.ccount.reserve(nc);
  w.foff.reserve(nc + 1);
  FB_LAUNCH(k_iso_masks, nblocks(n, 256), 256, 0, s, d_v, stride, L, out.iso, w.mask.p);
  scan_counts(NodeVertices{w.mask.p, n}, n, w.voff.p, w, s);
  FB_LAUNCH(k_iso_cube_counts, nblocks(nc, 256), 256, 0, s, w.mask.p, L, w.ccount.p);
  scan_counts(CubeFaces{w.ccount.p, nc}, nc, w.foff.p, w, s);
  unsigned long long tot[4] = {0, 0, 0, 0};
  FB_CUDA(cudaMemcpyAsync(&tot[0], w.voff.p + n, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
  FB_CUDA(cudaMemcpyAsync(&tot[1], w.foff.p + nc, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
  if (solid) {
    w.coff.reserve(nb + 1);
    w.scount.reserve(ns);
    w.soff.reserve(ns + 1);
    scan_counts(CapNodes{w.mask.p, L, side, nb}, nb, w.coff.p, w, s);
    FB_LAUNCH(k_iso_cap_counts, nblocks(ns, 256), 256, 0, s, w.mask.p, L, S, side, w.scount.p);
    scan_counts(CubeFaces{w.scount.p, ns}, ns, w.soff.p, w, s);
    FB_CUDA(cudaMemcpyAsync(&tot[2], w.coff.p + nb, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    FB_CUDA(cudaMemcpyAsync(&tot[3], w.soff.p + ns, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
  }
  FB_CUDA(cudaStreamSynchronize(s));
  out.nv = tot[0];
  out.nf = tot[1];
  out.cv = tot[2];
  out.cf = tot[3];
  if (out.nv + out.cv) out.verts.reserve(3 * (out.nv + out.cv));
  if (out.nv) {
    out.edge.reserve(out.nv);
    FB_LAUNCH(k_iso_vertices, nblocks(n, 256), 256, 0, s, d_v, stride, L, out.iso, w.mask.p, w.voff.p, out.verts.p,
              out.edge.p);
  }
  if (out.cv) {
    out.cap_node.reserve(out.cv);
    FB_LAUNCH(k_iso_cap_nodes, nblocks(nb, 256), 256, 0, s, w.mask.p, L, side, w.coff.p, out.nv, out.verts.p,
              out.cap_node.p);
  }
  if (out.nf + out.cf) out.faces.reserve(3 * (out.nf + out.cf));
  if (out.nf)
    FB_LAUNCH(k_iso_triangles, nblocks(nc, 256), 256, 0, s, w.mask.p, L, w.voff.p, w.foff.p, solid && side == 1,
              out.faces.p);
  if (out.cf)
    FB_LAUNCH(k_iso_cap_faces, nblocks(ns, 256), 256, 0, s, w.mask.p, L, S, side, w.voff.p, w.coff.p, w.soff.p, out.nv,
              out.nf, out.faces.p);
}

void iso_refine(const double *d_v, size_t stride, const IsoLattice &L, int n_cols, int col, const IsoEval &eval,
                IsoScratch &w, IsoSurface &surf, cudaStream_t s) {
  surf.evaluations = surf.max_iterations = 0;
  const uint64_t nv = surf.nv;
  if (!nv) return;
  w.state.reserve(nv);
  w.act[0].reserve(nv);
  w.act[1].reserve(nv);
  w.keep.reserve(nv);
  w.pts.reserve(3 * nv);
  w.vals.reserve(nv * (size_t)n_cols);
  w.n_sel.reserve(1);
  FB_LAUNCH(k_iso_refine_init, nblocks(nv, 256), 256, 0, s, d_v, stride, L, surf.iso, surf.edge.p, nv, w.state.p,
            w.act[0].p);
  uint64_t na = nv;
  int cur = 0;
  while (na > 0) {
    FB_LAUNCH(k_iso_refine_points, nblocks(na, 256), 256, 0, s, L, surf.edge.p, w.state.p, w.act[cur].p, na, w.pts.p);
    eval(w.pts.p, na, w.vals.p);
    FB_LAUNCH(k_iso_refine_update, nblocks(na, 256), 256, 0, s, w.vals.p, n_cols, col, surf.iso, w.act[cur].p, na,
              w.pts.p, w.state.p, surf.verts.p, w.keep.p);
    surf.evaluations += na;
    ++surf.max_iterations;
    size_t bytes = 0;
    FB_CUDA(cub::DeviceSelect::Flagged(nullptr, bytes, w.act[cur].p, w.keep.p, w.act[cur ^ 1].p, w.n_sel.p, (int)na, s));
    w.cub.reserve(bytes);
    FB_CUDA(cub::DeviceSelect::Flagged(w.cub.p, bytes, w.act[cur].p, w.keep.p, w.act[cur ^ 1].p, w.n_sel.p, (int)na, s));
    g_launches.fetch_add(1);
    int h = 0;
    FB_CUDA(cudaMemcpyAsync(&h, w.n_sel.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    FB_CUDA(cudaStreamSynchronize(s));
    na = (uint64_t)h;
    cur ^= 1;
  }
}

void iso_normals(const double *d_grads, int n_cols, int col, const IsoLattice &L, IsoSurface &surf, cudaStream_t s) {
  surf.has_normals = true;
  if (!surf.nv && !surf.cv) return;
  surf.normals.reserve(3 * (surf.nv + surf.cv));
  if (surf.nv)
    FB_LAUNCH(k_iso_normals, nblocks(surf.nv, 256), 256, 0, s, d_grads, n_cols, col, surf.nv, surf.side == 1,
              surf.normals.p);
  if (surf.cv)
    FB_LAUNCH(k_iso_cap_normals, nblocks(surf.cv, 256), 256, 0, s, L, surf.cap_node.p, surf.cv,
              surf.normals.p + 3 * surf.nv);
}

void iso_measure(const IsoLattice &L, IsoScratch &w, IsoSurface &surf, cudaStream_t s) {
  w.sums.reserve(2);
  FB_CUDA(cudaMemsetAsync(w.sums.p, 0, 2 * sizeof(double), s));
  if (surf.nf + surf.cf)  // relative to the lattice's lo corner: at UTM coordinates the products would cancel
    reduce_sum(FaceVolume{surf.verts.p, surf.faces.p, {L.lo[0], L.lo[1], L.lo[2]}}, surf.nf + surf.cf, w.sums.p, w, s);
  if (surf.nf) reduce_sum(FaceArea{surf.verts.p, surf.faces.p}, surf.nf, w.sums.p + 1, w, s);
  double h[2] = {0, 0};
  FB_CUDA(cudaMemcpyAsync(h, w.sums.p, sizeof(h), cudaMemcpyDeviceToHost, s));
  FB_CUDA(cudaStreamSynchronize(s));
  surf.volume = h[0] / 6.0;
  surf.area = 0.5 * h[1];
}

}  // namespace fb

using namespace fb;

// ------------------------------------------------------------------------------------------ C ABI
namespace {
const IsoSurface &surface_of(const fr_isosurface *h, int which) {
  FB_REQUIRE(h, "null isosurface handle");
  FB_REQUIRE(which >= 0 && (size_t)which < h->surf.size(),
             "which must name one of the handle's " + std::to_string(h->surf.size()) + " isosurfaces");
  return *h->surf[which];
}
}  // namespace

namespace {
// the mesh of fr_lattice_isosurface (side kIsoOpen) or the solid of fr_lattice_solid
void lattice_mesh(const double *d_values, const uint64_t *resolution, const double *extents, double isovalue, int side,
                  void *stream, fr_isosurface **out) {
  FB_REQUIRE(out, "output handle required");
  *out = nullptr;
  FB_REQUIRE(d_values, "values must be an nz x ny x nx device array");
  const IsoLattice L = iso_lattice(extents, resolution);
  FB_REQUIRE(std::isfinite(isovalue), "isovalue must be finite");
  int device = 0;
  FB_CUDA(cudaGetDevice(&device));
  require_device_matrix(d_values, L.nodes(), 1, 1, 1, device, "values");
  const auto t0 = std::chrono::steady_clock::now();
  auto h = std::make_unique<fr_isosurface>();
  h->device = device;
  const cudaStream_t s = (cudaStream_t)stream;
  IsoScratch w;
  const uint64_t bad = iso_first_nonfinite(d_values, 1, L.nodes(), w, s);
  FB_REQUIRE(bad == L.nodes(), "lattice value " + std::to_string(bad) + " is not finite");
  h->surf.push_back(std::make_unique<IsoSurface>());
  h->surf[0]->iso = isovalue;
  h->surf[0]->side = side;
  iso_extract(d_values, 1, L, w, *h->surf[0], s);
  if (side != kIsoOpen) iso_measure(L, w, *h->surf[0], s);
  FB_CUDA(cudaStreamSynchronize(s));
  h->ms[1] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  *out = h.release();
}
}  // namespace

extern "C" {

int fr_lattice_isosurface(const double *d_values, const uint64_t *resolution, const double *extents, double isovalue,
                          void *stream, fr_isosurface **out) {
  return guarded([&] { lattice_mesh(d_values, resolution, extents, isovalue, kIsoOpen, stream, out); });
}

int fr_lattice_solid(const double *d_values, const uint64_t *resolution, const double *extents, double isovalue,
                     int side, void *stream, fr_isosurface **out) {
  return guarded([&] {
    if (out) *out = nullptr;
    FB_REQUIRE(side == 0 || side == 1, "side must be 0 (below) or 1 (above)");
    lattice_mesh(d_values, resolution, extents, isovalue, side, stream, out);
  });
}

int fr_isosurface_counts(const fr_isosurface *s, int which, uint64_t *n_vertices, uint64_t *n_faces) {
  return guarded([&] {
    const IsoSurface &f = surface_of(s, which);
    if (n_vertices) *n_vertices = f.nv + f.cv;
    if (n_faces) *n_faces = f.nf + f.cf;
  });
}

int fr_isosurface_copy(const fr_isosurface *s, int which, double *vertices, int64_t *faces, double *normals_or_null) {
  return guarded([&] {
    const IsoSurface &f = surface_of(s, which);
    const uint64_t nv = f.nv + f.cv, nf = f.nf + f.cf;
    FB_REQUIRE((vertices || !nv) && (faces || !nf), "vertices and faces outputs are required");
    FB_REQUIRE(!normals_or_null || f.has_normals, "this isosurface has no normals: lattice values carry no gradient");
    FB_CUDA(cudaSetDevice(s->device));
    if (nv) FB_CUDA(cudaMemcpy(vertices, f.verts.p, 3 * nv * sizeof(double), cudaMemcpyDefault));
    if (nf) FB_CUDA(cudaMemcpy(faces, f.faces.p, 3 * nf * sizeof(int64_t), cudaMemcpyDefault));
    if (normals_or_null && nv)
      FB_CUDA(cudaMemcpy(normals_or_null, f.normals.p, 3 * nv * sizeof(double), cudaMemcpyDefault));
  });
}

int fr_isosurface_solid_info(const fr_isosurface *s, int which, uint64_t *surface_vertices, uint64_t *surface_faces,
                             double *volume, double *surface_area) {
  return guarded([&] {
    const IsoSurface &f = surface_of(s, which);
    FB_REQUIRE(f.side != kIsoOpen, "this handle holds open isosurfaces, not solids");
    if (surface_vertices) *surface_vertices = f.nv;
    if (surface_faces) *surface_faces = f.nf;
    if (volume) *volume = f.volume;
    if (surface_area) *surface_area = f.area;
  });
}

int fr_isosurface_timing(const fr_isosurface *s, double *ms_out4) {
  return guarded([&] {
    FB_REQUIRE(s && ms_out4, "handle and output required");
    std::copy(s->ms, s->ms + 4, ms_out4);
  });
}

int fr_isosurface_refine_stats(const fr_isosurface *s, int which, uint64_t *evaluations, uint64_t *iterations) {
  return guarded([&] {
    const IsoSurface &f = surface_of(s, which);
    if (evaluations) *evaluations = f.evaluations;
    if (iterations) *iterations = f.max_iterations;
  });
}

void fr_isosurface_free(fr_isosurface *s) {
  if (!s) return;
  cudaSetDevice(s->device);
  delete s;
}

}  // extern "C"

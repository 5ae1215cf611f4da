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

struct CubeFaces {
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

__global__ void k_iso_triangles(const uint8_t *__restrict__ mask, IsoLattice L,
                                const unsigned long long *__restrict__ voff, const unsigned long long *__restrict__ foff,
                                long long *__restrict__ faces) {
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
      const bool swap = (kSwap[pi] >> (2 * m + t)) & 1u;
      faces[3 * f] = vid[0];
      faces[3 * f + 1] = swap ? vid[2] : vid[1];
      faces[3 * f + 2] = swap ? vid[1] : vid[2];
      ++f;
    }
  }
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

__global__ void k_iso_normals(const double *__restrict__ g, int n_cols, int col, uint64_t nv,
                              double *__restrict__ nrm) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= nv) return;
  const double *gi = g + i * (uint64_t)(3 * n_cols) + 3 * col;
  const double x = gi[0], y = gi[1], z = gi[2];
  const double len = sqrt(x * x + y * y + z * z);
  const double inv = len > 0.0 ? 1.0 / len : 0.0;
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
  w.mask.reserve(n);
  w.voff.reserve(n + 1);
  w.ccount.reserve(nc);
  w.foff.reserve(nc + 1);
  FB_LAUNCH(k_iso_masks, nblocks(n, 256), 256, 0, s, d_v, stride, L, out.iso, w.mask.p);
  scan_counts(NodeVertices{w.mask.p, n}, n, w.voff.p, w, s);
  FB_LAUNCH(k_iso_cube_counts, nblocks(nc, 256), 256, 0, s, w.mask.p, L, w.ccount.p);
  scan_counts(CubeFaces{w.ccount.p, nc}, nc, w.foff.p, w, s);
  unsigned long long tot[2] = {0, 0};
  FB_CUDA(cudaMemcpyAsync(&tot[0], w.voff.p + n, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
  FB_CUDA(cudaMemcpyAsync(&tot[1], w.foff.p + nc, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
  FB_CUDA(cudaStreamSynchronize(s));
  out.nv = tot[0];
  out.nf = tot[1];
  if (out.nv) {
    out.verts.reserve(3 * out.nv);
    out.edge.reserve(out.nv);
    FB_LAUNCH(k_iso_vertices, nblocks(n, 256), 256, 0, s, d_v, stride, L, out.iso, w.mask.p, w.voff.p, out.verts.p,
              out.edge.p);
  }
  if (out.nf) {
    out.faces.reserve(3 * out.nf);
    FB_LAUNCH(k_iso_triangles, nblocks(nc, 256), 256, 0, s, w.mask.p, L, w.voff.p, w.foff.p, out.faces.p);
  }
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

void iso_normals(const double *d_grads, int n_cols, int col, IsoSurface &surf, cudaStream_t s) {
  surf.has_normals = true;
  if (!surf.nv) return;
  surf.normals.reserve(3 * surf.nv);
  FB_LAUNCH(k_iso_normals, nblocks(surf.nv, 256), 256, 0, s, d_grads, n_cols, col, surf.nv, surf.normals.p);
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

extern "C" {

int fr_lattice_isosurface(const double *d_values, const uint64_t *resolution, const double *extents, double isovalue,
                          void *stream, fr_isosurface **out) {
  return guarded([&] {
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
    iso_extract(d_values, 1, L, w, *h->surf[0], s);
    FB_CUDA(cudaStreamSynchronize(s));
    h->ms[1] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    *out = h.release();
  });
}

int fr_isosurface_counts(const fr_isosurface *s, int which, uint64_t *n_vertices, uint64_t *n_faces) {
  return guarded([&] {
    const IsoSurface &f = surface_of(s, which);
    if (n_vertices) *n_vertices = f.nv;
    if (n_faces) *n_faces = f.nf;
  });
}

int fr_isosurface_copy(const fr_isosurface *s, int which, double *vertices, int64_t *faces, double *normals_or_null) {
  return guarded([&] {
    const IsoSurface &f = surface_of(s, which);
    FB_REQUIRE((vertices || !f.nv) && (faces || !f.nf), "vertices and faces outputs are required");
    FB_REQUIRE(!normals_or_null || f.has_normals, "this isosurface has no normals: lattice values carry no gradient");
    FB_CUDA(cudaSetDevice(s->device));
    if (f.nv) FB_CUDA(cudaMemcpy(vertices, f.verts.p, 3 * f.nv * sizeof(double), cudaMemcpyDefault));
    if (f.nf) FB_CUDA(cudaMemcpy(faces, f.faces.p, 3 * f.nf * sizeof(int64_t), cudaMemcpyDefault));
    if (normals_or_null && f.nv)
      FB_CUDA(cudaMemcpy(normals_or_null, f.normals.p, 3 * f.nv * sizeof(double), cudaMemcpyDefault));
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

"""Numpy restatement of the lattice solids of ``fr_lattice_solid`` / ``fr_isosurface_extract_solid``
(csrc/isosurface.cu), written from their specification (DESIGN.md, "Solids"): the isosurface of
tests/isosurface_oracle.py closed at the lattice box by caps built from the boundary nodes of the solid's side and the
existing rim vertices, oriented by a fixed table derived here on the unit square, and the volume and area of the
result.  Test infrastructure only."""
import numpy as np

from tests import isosurface_oracle as oi

SIDES = {"below": 0, "above": 1}


def face_axes(f):
    """(w, hi, u, v) of box face f = 0..5 (x lo, x hi, y lo, y hi, z lo, z hi): normal axis w, in-plane axes u < v"""
    w, hi = f // 2, f % 2
    u, v = [d for d in range(3) if d != w]
    return w, hi, u, v


# triangles of a lattice square with minimum corner a, as 0/1 offsets along (u, v): T0 = (a, a + e_u, a + e_u + e_v),
# T1 = (a, a + e_v, a + e_u + e_v)
SQUARE_TRIANGLES = (((0, 0), (1, 0), (1, 1)), ((0, 0), (0, 1), (1, 1)))


def clip(mask):
    """sub-triangles of a triangle whose inside corners (positions 0..2) are the set bits of `mask`; an entry is a
    corner position q or an edge (q, r) between positions"""
    inside = [q for q in range(3) if (mask >> q) & 1]
    out = [q for q in range(3) if not (mask >> q) & 1]
    if len(inside) == 1:
        q, (r1, r2) = inside[0], out
        return [[q, (q, r1), (q, r2)]]
    if len(inside) == 2:
        (q1, q2), r = inside, out[0]
        return [[q1, q2, (q2, r)], [q1, (q2, r), (q1, r)]]
    if len(inside) == 3:
        return [[0, 1, 2]]
    return []


def cap_swap_table():
    """swap[face][tri][mask][sub]: True where the sub-triangle's last two vertices are exchanged so that (B-A) x (C-A)
    points out of the box.  Decided on the unit square with the crossing points at edge midpoints, so it depends on
    (face, tri, mask, sub) alone."""
    table = np.zeros((6, 2, 8, 2), dtype=bool)
    for f in range(6):
        w, hi, u, v = face_axes(f)
        out = np.zeros(3)
        out[w] = 1.0 if hi else -1.0
        for t, tri in enumerate(SQUARE_TRIANGLES):
            c = []
            for ou, ov in tri:
                x = np.zeros(3)
                x[u], x[v] = ou, ov
                c.append(x)
            for mask in range(1, 8):
                for s, sub in enumerate(clip(mask)):
                    a, b, d = [c[e] if isinstance(e, int) else 0.5 * (c[e[0]] + c[e[1]]) for e in sub]
                    g = float(np.dot(np.cross(b - a, d - a), out))
                    assert g != 0.0
                    table[f, t, mask, s] = g < 0
    return table


def crossing_edge_ids(values, iso):
    """sorted edge ids 7 p(a) + mask - 1 of the crossing edges: vertex k of the isosurface lies on edge ids[k]"""
    v = np.asarray(values, dtype=np.float64)
    nz, ny, nx = v.shape
    below = v.ravel() < iso
    k, j, i = [g.ravel() for g in np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")]
    p = np.arange(below.size, dtype=np.int64)
    ids = []
    for m in range(1, 8):
        s = (m & 1, (m >> 1) & 1, m >> 2)
        ok = (i + s[0] < nx) & (j + s[1] < ny) & (k + s[2] < nz)
        a = p[ok]
        b = a + s[0] + nx * (s[1] + ny * s[2])
        ids.append(7 * a[below[a] != below[b]] + (m - 1))
    return np.sort(np.concatenate(ids))


def extract_solid(values, extents, iso, side="below"):
    """(vertices (V, 3), faces (F, 3) int64, n_surface_vertices, n_surface_faces) of the solid {f < iso} ("below") or
    {f >= iso} ("above") of lattice values (nz, ny, nx), closed at the lattice box"""
    sd = SIDES[side]
    v = np.asarray(values, dtype=np.float64)
    nz, ny, nx = v.shape
    n = (nx, ny, nz)
    sv, sf = oi.extract(v, extents, iso)
    if sd == 1:
        sf = sf[:, [0, 2, 1]]
    nvs = sv.shape[0]
    ids = crossing_edge_ids(v, iso)
    inside = (v.ravel() < iso) if sd == 0 else ~(v.ravel() < iso)

    k, j, i = [g.ravel() for g in np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")]
    on_box = (i == 0) | (i == nx - 1) | (j == 0) | (j == ny - 1) | (k == 0) | (k == nz - 1)
    cap_nodes = np.flatnonzero(on_box & inside)          # ascending node index
    cap_id = np.full(v.size, -1, dtype=np.int64)
    cap_id[cap_nodes] = nvs + np.arange(cap_nodes.size)
    verts = np.concatenate([sv, oi.lattice_points(extents, n)[cap_nodes]])

    table = cap_swap_table()
    keys, faces = [], []
    for f in range(6):
        w, hi, u, v_ = face_axes(f)
        nu, nv = n[u], n[v_]
        av, au = [g.ravel() for g in np.meshgrid(np.arange(nv - 1), np.arange(nu - 1), indexing="ij")]
        square = au + (nu - 1) * av
        idx = [None, None, None]
        idx[u], idx[v_], idx[w] = au, av, np.full(au.shape, n[w] - 1 if hi else 0)
        base = idx[0] + nx * (idx[1] + ny * idx[2])

        def node(ou, ov):
            off = [0, 0, 0]
            off[u], off[v_] = ou, ov
            return base + off[0] + nx * (off[1] + ny * off[2]), off

        for t, tri in enumerate(SQUARE_TRIANGLES):
            c = [node(ou, ov) for ou, ov in tri]
            mask = sum(inside[c[q][0]].astype(np.int64) << q for q in range(3))
            for m in range(1, 8):
                sel = mask == m
                if not sel.any():
                    continue
                for s, sub in enumerate(clip(m)):
                    fc = np.empty((int(sel.sum()), 3), dtype=np.int64)
                    for col, e in enumerate(sub):
                        if isinstance(e, int):
                            fc[:, col] = cap_id[c[e][0][sel]]
                        else:
                            lo, hi_ = min(e), max(e)
                            d = np.array(c[hi_][1]) - np.array(c[lo][1])
                            eid = 7 * c[lo][0][sel] + int(d[0] + 2 * d[1] + 4 * d[2]) - 1
                            fc[:, col] = np.searchsorted(ids, eid)
                    if table[f, t, m, s]:
                        fc[:, [1, 2]] = fc[:, [2, 1]]
                    faces.append(fc)
                    keys.append(np.stack([np.full(fc.shape[0], f), square[sel], np.full(fc.shape[0], t),
                                          np.full(fc.shape[0], s)], axis=1))
    if faces:
        cf = np.concatenate(faces)
        kk = np.concatenate(keys)
        cf = cf[np.lexsort((kk[:, 3], kk[:, 2], kk[:, 1], kk[:, 0]))]
    else:
        cf = np.zeros((0, 3), dtype=np.int64)
    return verts, np.concatenate([sf, cf]), nvs, sf.shape[0]


def volume(verts, faces, origin):
    """(1/6) sum over faces of det(A - o, B - o, C - o)"""
    x = np.asarray(verts) - np.asarray(origin, dtype=np.float64)
    f = np.asarray(faces)
    if not len(f):
        return 0.0
    return float(np.einsum("ij,ij->i", x[f[:, 0]], np.cross(x[f[:, 1]], x[f[:, 2]])).sum() / 6.0)


def clip_volume(values, extents, iso, side="below"):
    """volume of the sublevel (superlevel) set of the piecewise-linear interpolant over the Kuhn tetrahedra: per
    tetrahedron the convex hull of its inside corners and its crossing points, independent of the mesh"""
    from scipy.spatial import ConvexHull
    v = np.asarray(values, dtype=np.float64)
    nz, ny, nx = v.shape
    x = oi.lattice_points(extents, (nx, ny, nz))
    flat = v.ravel()
    inside = (flat < iso) if side == "below" else ~(flat < iso)
    total = 0.0
    for k in range(nz - 1):
        for j in range(ny - 1):
            for i in range(nx - 1):
                base = i + nx * (j + ny * k)
                for pi in oi.PERMS:
                    nodes = [base + o[0] + nx * (o[1] + ny * o[2]) for o in oi.chain(pi)]
                    ins = [q for q in range(4) if inside[nodes[q]]]
                    if not ins:
                        continue
                    pts = [x[nodes[q]] for q in ins]
                    for q in ins:
                        for r in range(4):
                            if r not in ins:
                                a, b = nodes[q], nodes[r]
                                t = (iso - flat[a]) / (flat[b] - flat[a])
                                pts.append(x[a] + t * (x[b] - x[a]))
                    total += ConvexHull(np.array(pts)).volume
    return total

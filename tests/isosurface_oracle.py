"""Numpy restatement of the lattice isosurface of ``fr_lattice_isosurface`` (csrc/isosurface.cu), written from its
specification (DESIGN.md, "Isosurfaces"): the lattice of ``np.linspace`` nodes, the six Kuhn tetrahedra per cube,
one vertex per crossing edge numbered by edge id, and triangles oriented by a fixed table derived here from the
geometry of the unit cube.  Test infrastructure only: vectorised per tetrahedron class, not per cube."""
import numpy as np

# permutations of (x, y, z) in lexicographic order: tetrahedron pi of a cube with minimum corner c is the chain
# c, c + e[pi0], c + e[pi0] + e[pi1], c + (1, 1, 1)
PERMS = ((0, 1, 2), (0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1), (2, 1, 0))


def axes(extents, resolution):
    """per axis: node idx * step + lo with step = (hi - lo) / (n - 1), the last node exactly hi"""
    ext = np.asarray(extents, dtype=np.float64)
    out = []
    for d in range(3):
        n, lo, hi = int(resolution[d]), ext[d], ext[3 + d]
        step = (hi - lo) / (n - 1)
        a = np.arange(n, dtype=np.float64) * step + lo
        a[-1] = hi
        out.append(a)
    return out


def lattice_points(extents, resolution):
    """(nx * ny * nz, 3) node coordinates, node p = i + nx * (j + ny * k)"""
    ax, ay, az = axes(extents, resolution)
    z, y, x = np.meshgrid(az, ay, ax, indexing="ij")
    return np.stack([x.ravel(), y.ravel(), z.ravel()], axis=1)


def chain(pi):
    """the 4 corners of tetrahedron pi as 0/1 offsets from the cube's minimum corner"""
    c = [np.zeros(3, dtype=np.int64)]
    for d in pi:
        nxt = c[-1].copy()
        nxt[d] += 1
        c.append(nxt)
    return c


def triangles_of(mask):
    """triangles (as chain-position pairs) of a tetrahedron whose below corners are the set bits of `mask`"""
    below = [q for q in range(4) if (mask >> q) & 1]
    above = [q for q in range(4) if not (mask >> q) & 1]
    if len(below) in (1, 3):
        q = below[0] if len(below) == 1 else above[0]
        r = [x for x in range(4) if x != q]
        return [[(q, r[0]), (q, r[1]), (q, r[2])]]
    if len(below) == 2:
        a, b = below
        c, d = above
        return [[(a, c), (a, d), (b, d)], [(a, c), (b, d), (b, c)]]
    return []


def swap_table():
    """swap[pi][mask][tri]: True where the triangle's last two vertices are exchanged so that (B-A) x (C-A) points
    from the below corners to the others.  Decided on the edge midpoints of the unit cube, so it depends on
    (pi, mask, tri) alone."""
    table = np.zeros((6, 16, 2), dtype=bool)
    for p, pi in enumerate(PERMS):
        ch = [c.astype(np.float64) for c in chain(pi)]
        for mask in range(1, 15):
            bel = np.mean([ch[q] for q in range(4) if (mask >> q) & 1], axis=0)
            abv = np.mean([ch[q] for q in range(4) if not (mask >> q) & 1], axis=0)
            for t, tri in enumerate(triangles_of(mask)):
                a, b, c = [0.5 * (ch[u] + ch[w]) for u, w in tri]
                s = float(np.dot(np.cross(b - a, c - a), abv - bel))
                assert s != 0.0
                table[p, mask, t] = s < 0
    return table


def extract(values, extents, iso):
    """(vertices (V, 3) float64, faces (F, 3) int64) of the level set `iso` of lattice values (nz, ny, nx)"""
    v = np.asarray(values, dtype=np.float64)
    nz, ny, nx = v.shape
    res = (nx, ny, nz)
    flat = v.ravel()
    below = flat < iso
    ax = axes(extents, res)
    k, j, i = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    i, j, k = i.ravel(), j.ravel(), k.ravel()
    p = np.arange(flat.size, dtype=np.int64)

    # crossing edges a -> a + s, s a nonzero 0/1 vector with mask sx + 2 sy + 4 sz, edge id 7 p(a) + mask - 1
    ids, pos = [], []
    for m in range(1, 8):
        s = np.array([m & 1, (m >> 1) & 1, (m >> 2) & 1])
        ok = (i + s[0] < nx) & (j + s[1] < ny) & (k + s[2] < nz)
        a = p[ok]
        b = a + s[0] + nx * (s[1] + ny * s[2])
        cr = below[a] != below[b]
        a, b = a[cr], b[cr]
        va, vb = flat[a], flat[b]
        t = (iso - va) / (vb - va)
        xyz = np.empty((a.size, 3))
        for d, idx in enumerate((i, j, k)):
            xa = ax[d][idx[a]]
            xb = ax[d][idx[b]]
            xyz[:, d] = xa + t * (xb - xa)
        ids.append(7 * a + (m - 1))
        pos.append(xyz)
    ids = np.concatenate(ids)
    pos = np.concatenate(pos)
    order = np.argsort(ids, kind="stable")
    ids, verts = ids[order], pos[order]

    # triangles, ordered by (cube index, pi, triangle)
    cx, cy, cz = nx - 1, ny - 1, nz - 1
    ck, cj, ci = [g.ravel() for g in np.meshgrid(np.arange(cz), np.arange(cy), np.arange(cx), indexing="ij")]
    cube = np.arange(cx * cy * cz, dtype=np.int64)
    base = ci + nx * (cj + ny * ck)
    table = swap_table()
    keys, faces = [], []
    for t_pi, pi in enumerate(PERMS):
        ch = chain(pi)
        node = [base + o[0] + nx * (o[1] + ny * o[2]) for o in ch]
        mask = sum(below[node[q]].astype(np.int64) << q for q in range(4))
        for m in range(1, 15):
            sel = mask == m
            if not sel.any():
                continue
            for t, tri in enumerate(triangles_of(m)):
                f = np.empty((int(sel.sum()), 3), dtype=np.int64)
                for c, (u, w) in enumerate(tri):
                    lo, hi = min(u, w), max(u, w)
                    s = ch[hi] - ch[lo]
                    eid = 7 * node[lo][sel] + (int(s[0] + 2 * s[1] + 4 * s[2]) - 1)
                    f[:, c] = np.searchsorted(ids, eid)
                if table[t_pi, m, t]:
                    f[:, [1, 2]] = f[:, [2, 1]]
                faces.append(f)
                keys.append(np.stack([cube[sel], np.full(f.shape[0], t_pi), np.full(f.shape[0], t)], axis=1))
    if not faces:
        return verts, np.zeros((0, 3), dtype=np.int64)
    faces = np.concatenate(faces)
    keys = np.concatenate(keys)
    order = np.lexsort((keys[:, 2], keys[:, 1], keys[:, 0]))
    return verts, faces[order]


# ---- measures of a mesh, for the tests -------------------------------------------------------------------------------
def directed_edges(faces):
    f = np.asarray(faces, dtype=np.int64)
    return np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])


def edge_use(faces):
    """(every directed edge occurs once, set of undirected edges used only once: the open boundary)"""
    de = directed_edges(faces)
    uniq, cnt = np.unique(de, axis=0, return_counts=True)
    once = bool((cnt == 1).all())
    key = {(int(a), int(b)) for a, b in uniq}
    open_edges = {(a, b) for a, b in key if (b, a) not in key}
    return once, open_edges


def euler_characteristic(verts, faces):
    de = directed_edges(faces)
    und = np.unique(np.sort(de, axis=1), axis=0)
    used = np.unique(np.asarray(faces).ravel()).size
    return used - und.shape[0] + len(faces)


def face_normals(verts, faces):
    v = np.asarray(verts)
    f = np.asarray(faces)
    return np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]])


def area(verts, faces):
    return 0.5 * float(np.linalg.norm(face_normals(verts, faces), axis=1).sum())

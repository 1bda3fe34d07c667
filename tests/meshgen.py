"""Procedural closed meshes: the bumpy torus standing in for the reference's missing dragon.obj / Ramesses.obj (SURVEY.md §8d,
F10), and small shapes with sharp edges, reflex edges, slivers, high valence, nested shells and non-manifold vertices.
Every mesh is closed and counter-clockwise seen from outside; its f32 vertices are the exact geometry."""
import numpy as np


def bumpy_torus(U=60, V=40):
    """Watertight 'bumpy torus' grid (SURVEY.md §8d C3): R = 0.30 + 0.03 sin(5u) cos(3v), r = 0.10 + 0.02 sin(7v + 2u).
    2 U V triangles, counter-clockwise seen from outside. U=1000, V=435 is the 870 k-triangle dragon stand-in,
    U=1000, V=800 the 1.6 M-triangle Ramesses stand-in."""
    u = (np.arange(U) * (2 * np.pi / U))[:, None]
    v = (np.arange(V) * (2 * np.pi / V))[None, :]
    R = 0.30 + 0.03 * np.sin(5 * u) * np.cos(3 * v)
    r = 0.10 + 0.02 * np.sin(7 * v + 2 * u)
    x = (R + r * np.cos(v)) * np.cos(u)
    y = (R + r * np.cos(v)) * np.sin(u)
    z = r * np.sin(v) + 0 * u
    verts = np.stack([x, y, z], -1).reshape(-1, 3).astype(np.float32)
    i, j = np.meshgrid(np.arange(U), np.arange(V), indexing="ij")
    a = (i * V + j).ravel()
    b = (((i + 1) % U) * V + j).ravel()
    c = (((i + 1) % U) * V + (j + 1) % V).ravel()
    d = (i * V + (j + 1) % V).ravel()
    tris = np.concatenate([np.stack([a, b, c], 1), np.stack([a, c, d], 1)]).astype(np.uint32)
    return verts, tris


def mesh_root(verts):
    """Root box of the mesh configs: AABB centre +- 0.6 * max extent (SURVEY.md §8d C3)."""
    mn, mx = verts.min(0).astype(np.float64), verts.max(0).astype(np.float64)
    c, e = (mn + mx) / 2, (mx - mn).max()
    return tuple((c - 0.6 * e).tolist()), tuple((c + 0.6 * e).tolist())


def box_mesh(k, half=0.3):
    """Closed axis-aligned cube, every face split into k x k squares of two triangles, counter-clockwise seen from outside:
    face normals ±x, ±y, ±z (the normal -z and the axis-aligned frames of the wide nodes)."""
    index, verts, tris = {}, [], []

    def vid(p):
        if p not in index:
            index[p] = len(verts)
            verts.append(p)
        return index[p]

    for a in range(3):
        b, c = (a + 1) % 3, (a + 2) % 3
        for side in (0, k):
            for i in range(k):
                for j in range(k):
                    q = []
                    for di, dj in ((0, 0), (1, 0), (1, 1), (0, 1)):
                        p = [0, 0, 0]
                        p[a], p[b], p[c] = side, i + di, j + dj
                        q.append(vid(tuple(p)))
                    if side == k:           # b x c = +a: counter-clockwise in (b, c) faces +a
                        tris += [(q[0], q[1], q[2]), (q[0], q[2], q[3])]
                    else:
                        tris += [(q[0], q[2], q[1]), (q[0], q[3], q[2])]
    v = (np.array(verts, np.float64) / k * 2 - 1) * half
    return v.astype(np.float32), np.array(tris, np.uint32)


def tetrahedron(s=0.3):
    """Closed mesh of 4 triangles: one BVH leaf, so the wide tree is the single-leaf root."""
    v = np.array([[1, 1, 1], [1, -1, -1], [-1, 1, -1], [-1, -1, 1]], np.float64) * s
    tris = []
    for f in ((0, 1, 2), (0, 1, 3), (0, 2, 3), (1, 2, 3)):
        other = ({0, 1, 2, 3} - set(f)).pop()
        a, b, c = v[list(f)]
        if np.dot(np.cross(b - a, c - a), a - v[other]) < 0:
            f = (f[0], f[2], f[1])
        tris.append(f)
    return v.astype(np.float32), np.array(tris, np.uint32)


def octahedron(s=0.3):
    """Regular octahedron |x| + |y| + |z| = s: 8 triangles, 90-degree vertices of valence 4."""
    v = np.array([[s, 0, 0], [-s, 0, 0], [0, s, 0], [0, -s, 0], [0, 0, s], [0, 0, -s]], np.float32)
    tris = []
    for x in (0, 1):
        for y in (2, 3):
            for z in (4, 5):
                f = [x, y, z]
                if np.linalg.det(v[f].astype(np.float64)) < 0:          # outward normal: the corner's octant sign
                    f = [x, z, y]
                tris.append(f)
    return v, np.array(tris, np.uint32)


def bipyramid(n, r=0.3, h=0.3):
    """n-gon bipyramid: a rim of n vertices on the circle of radius r at z = 0 and apexes at z = +-h. 2n triangles; the apexes
    have valence n (angles of 2 pi / n at n = 4096), the triangles are slivers for large n."""
    a = np.arange(n) * (2 * np.pi / n)
    rim = np.stack([r * np.cos(a), r * np.sin(a), np.zeros(n)], 1)
    v = np.concatenate([rim, [[0, 0, h], [0, 0, -h]]]).astype(np.float32)
    k = np.arange(n)
    k1 = (k + 1) % n
    top = np.stack([np.full(n, n), k, k1], 1)
    bottom = np.stack([np.full(n, n + 1), k1, k], 1)
    return v, np.concatenate([top, bottom]).astype(np.uint32)


def star_prism(points=5, r_out=0.3, r_in=0.12, h=0.1):
    """Prism over a star polygon (z in [-h, h]): reflex vertical edges at the inner corners, saddle vertices where they meet
    the caps. The caps are fans around a centre vertex."""
    m = 2 * points
    a = np.arange(m) * (2 * np.pi / m)
    r = np.where(np.arange(m) % 2 == 0, r_out, r_in)
    ring = np.stack([r * np.cos(a), r * np.sin(a)], 1)
    v = np.concatenate([np.concatenate([ring, np.full((m, 1), h)], 1), np.concatenate([ring, np.full((m, 1), -h)], 1),
                        [[0, 0, h], [0, 0, -h]]]).astype(np.float32)
    k = np.arange(m)
    k1 = (k + 1) % m
    top = np.stack([np.full(m, 2 * m), k, k1], 1)
    bottom = np.stack([np.full(m, 2 * m + 1), m + k1, m + k], 1)
    side = np.concatenate([np.stack([k, m + k, m + k1], 1), np.stack([k, m + k1, k1], 1)])
    return v, np.concatenate([top, bottom, side]).astype(np.uint32)


def icosphere(subdiv=2, r=0.3):
    """Sphere of 20 * 4^subdiv triangles: the icosahedron, each triangle split in four and projected to radius r."""
    g = (1 + 5 ** 0.5) / 2
    v = [[-1, g, 0], [1, g, 0], [-1, -g, 0], [1, -g, 0], [0, -1, g], [0, 1, g], [0, -1, -g], [0, 1, -g],
         [g, 0, -1], [g, 0, 1], [-g, 0, -1], [-g, 0, 1]]
    v = [list(np.array(p) / np.linalg.norm(p)) for p in v]
    f = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6), (7, 1, 8),
         (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10), (8, 6, 7), (9, 8, 1)]
    for _ in range(subdiv):
        mid, nf = {}, []

        def m(i, j):
            key = (min(i, j), max(i, j))
            if key not in mid:
                p = np.add(v[i], v[j])
                v.append(list(p / np.linalg.norm(p)))
                mid[key] = len(v) - 1
            return mid[key]
        for a, b, c in f:
            ab, bc, ca = m(a, b), m(b, c), m(c, a)
            nf += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        f = nf
    return (np.array(v) * r).astype(np.float32), np.array(f, np.uint32)


def hollow_ball(r_out=0.3, r_in=0.2, subdiv=2):
    """Two nested shells: an outer icosphere and an inverted inner one (its normals point into the cavity)."""
    vo, to = icosphere(subdiv, r_out)
    vi, ti = icosphere(subdiv, r_in)
    return np.concatenate([vo, vi]), np.concatenate([to, ti[:, ::-1] + len(vo)]).astype(np.uint32)


def tetrahedra_sharing_vertex(s=0.3):
    """The tetrahedron and its point reflection through its vertex 0: two solids touching at one non-manifold vertex, every
    edge still has exactly two half-edges."""
    v, t = tetrahedron(s)
    v2 = 2 * v[0] - v[1:]
    t2 = np.where(t == 0, 0, t + 3)[:, ::-1]            # the reflection reverses orientation
    return np.concatenate([v, v2]).astype(np.float32), np.concatenate([t, t2]).astype(np.uint32)


def thin_plate():
    """A 200 x 200 x 1 box: the two large faces have opposite normals in every BVH node above the leaves."""
    v, t = box_mesh(1, 1.0)
    return (v * np.float32([0.25, 0.25, 0.00125])).astype(np.float32), t


# Small shapes at the scale of the root box (edges of about 0.1 to 0.6), as the workloads use them.
SHAPES = {
    "cube": lambda: box_mesh(1),
    "cube_k3": lambda: box_mesh(3),
    "octahedron": octahedron,
    "star_prism": star_prism,
    "bipyramid_4096": lambda: bipyramid(4096),
    **{"bipyramid_%d" % n: (lambda n=n: bipyramid(n)) for n in range(3, 10)},
    "thin_plate": thin_plate,
    "hollow_ball": hollow_ball,
    "tetrahedra_sharing_vertex": tetrahedra_sharing_vertex,
    "cube_at_4096": lambda: ((box_mesh(1, 2.0)[0] + np.float32(4096)).astype(np.float32), box_mesh(1)[1]),
    "cube_1000": lambda: box_mesh(1, 1000.0),
    "torus": lambda: bumpy_torus(60, 40),
}

# Scale (a power of two, so the f32 vertices stay exact) at which the reference's absolute EPS = 1e-6 of ClosestSimplexToPt is
# below f32 resolution for every shape of SHAPES: see eps_reach.
EXACT_SCALE = 256.0


def scaled(mesh, s):
    v, t = mesh
    return (v * np.float32(s)).astype(np.float32), t


def eps_reach(v, t, eps=1e-6):
    """How far from an edge line the reference's region tests still call a point an edge point, as a fraction of the mesh
    size: EPS / (shortest edge * twice the smallest triangle area) / size (ClosestSimplexToPt compares products of lengths
    of degree 2 and 4 with EPS). At 1e-7 or less it is below f32 resolution."""
    V = v.astype(np.float64)
    A, B, C = V[t[:, 0]], V[t[:, 1]], V[t[:, 2]]
    ell = min(np.linalg.norm(B - A, axis=1).min(), np.linalg.norm(C - B, axis=1).min(), np.linalg.norm(A - C, axis=1).min())
    area2 = np.linalg.norm(np.cross(B - A, C - A), axis=1).min()
    return eps / (ell * area2) / (V.max(0) - V.min(0)).max()


def point_sets(v, t, rng, n_uniform=2000, n_features=300):
    """Query points of every class for one mesh, as f32 arrays by name:
    uniform  in the root box (mesh_root);
    far      10 and 1000 mesh sizes away from the centre, in all octants;
    on       exactly on vertices, and (to f32 rounding) on edge midpoints and face centroids;
    (each feature class takes at most n_features features, chosen at random)
    face / edge / vertex  along the face normal, the edge bisector and the angle-weighted vertex normal, at +-1e-1 .. +-1e-6
             of the mesh size: both sides of the surface, closest feature that face, edge or vertex;
    symmetry on the planes through the centre of the bounding box, on its axes and at the centre, where ties occur;
    ties     1 and 8 ulps from a vertex along +-e_i +-e_j: where the vertex's pseudonormal has two components of equal
             magnitude (a cube's corner) the f32 dot product with it cancels exactly, so the sign hangs on its last bits;
    medial   along the inward and outward bisectors of edges and vertices, 1e-2 .. 3e-1 of the size in: near the medial
             axis of concave and convex corners."""
    from mesh_exact import pseudonormals
    V = v.astype(np.float64)
    lo, hi = V.min(0), V.max(0)
    c, size = (lo + hi) / 2, (hi - lo).max()
    fn, edges, en, vn = pseudonormals(v, t)
    cen = V[t.astype(np.int64)].mean(1)
    mid = V[edges].mean(1)

    def pick(n):
        return rng.choice(n, min(n, n_features), replace=False)

    steps = np.array([1e-1, 1e-2, 1e-3, 1e-4, 1e-5, 1e-6])

    def offsets(base, dirs):
        s = size * steps[rng.integers(0, len(steps), len(base))] * rng.choice([-1.0, 1.0], len(base))
        return base + dirs * s[:, None]
    r0, r1 = (np.asarray(x) for x in mesh_root(v))
    octs = np.array([[sx, sy, sz] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)], np.float64)
    far = np.concatenate([c + f * size * (octs * (0.5 + rng.random((8, 3)))) for f in (10.0, 1000.0)])
    iv, ie, it = pick(len(V)), pick(len(edges)), pick(len(t))
    sym = rng.uniform(r0, r1, (300, 3))
    sym[:100, 0] = c[0]
    sym[100:200, 1] = c[1]
    sym[200:, 2] = c[2]
    axes = np.repeat(c[None], 30, 0)
    axes[np.arange(30), np.arange(30) % 3] += rng.uniform(-0.6, 0.6, 30) * size
    dirs = np.concatenate([en[ie], vn[iv]])
    base = np.concatenate([mid[ie], V[iv]])
    depth = size * 10.0 ** rng.uniform(-2, np.log10(0.3), len(base)) * rng.choice([-1.0, 1.0], len(base))
    ulp = np.spacing(np.abs(v[iv[:50]]).max(1)).astype(np.float64)
    ties = [V[iv[:50]] + (ulp * 2.0 ** m)[:, None] * np.array(d, np.float64) for m in (0, 3)
            for d in ([1, 1, 0], [1, -1, 0], [-1, 1, 0], [-1, -1, 0], [0, 1, 1], [0, 1, -1], [0, -1, 1], [0, -1, -1],
                      [1, 0, 1], [1, 0, -1], [-1, 0, 1], [-1, 0, -1])]
    sets = dict(uniform=rng.uniform(r0, r1, (n_uniform, 3)), far=far, on=np.concatenate([V[iv], mid[ie], cen[it]]),
                face=offsets(cen[it], fn[it]), edge=offsets(mid[ie], en[ie]), vertex=offsets(V[iv], vn[iv]),
                symmetry=np.concatenate([sym, axes, c[None]]), ties=np.concatenate(ties), medial=base + dirs * depth[:, None])
    return {k: p.astype(np.float32) for k, p in sets.items()}

"""Small closed triangle meshes written as binary STL files for the tests (no reference fixture is copied)."""
import struct

import numpy as np


def write_binary_stl(path, triangles):
    tri = np.asarray(triangles, dtype=np.float32)
    n = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    nn = np.linalg.norm(n, axis=1, keepdims=True)
    rec = np.zeros(tri.shape[0], dtype=np.dtype([("n", "<f4", 3), ("v", "<f4", (3, 3)), ("a", "<u2")]))
    rec["n"] = np.where(nn > 0, n / np.where(nn > 0, nn, 1), n)
    rec["v"] = tri
    with open(path, "wb") as f:
        f.write(b"s3b200 test mesh".ljust(80, b" "))
        f.write(struct.pack("<I", tri.shape[0]))
        f.write(rec.tobytes())


def cube_triangles(lo=(0.0, 0.0, 0.0), hi=(1.0, 1.0, 1.0)):
    x0, y0, z0 = lo
    x1, y1, z1 = hi
    v = np.array([[x0, y0, z0], [x1, y0, z0], [x1, y1, z0], [x0, y1, z0],
                  [x0, y0, z1], [x1, y0, z1], [x1, y1, z1], [x0, y1, z1]])
    quads = [(0, 3, 2, 1), (4, 5, 6, 7), (0, 1, 5, 4), (2, 3, 7, 6), (1, 2, 6, 5), (0, 4, 7, 3)]
    tris = []
    for a, b, c, d in quads:
        tris.append([v[a], v[b], v[c]])
        tris.append([v[a], v[c], v[d]])
    return np.array(tris)


def icosphere_triangles(subdivisions=2, radius=1.0, center=(0.0, 0.0, 0.0)):
    t = (1.0 + 5.0 ** 0.5) / 2.0
    verts = [(-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t),
             (t, 0, -1), (t, 0, 1), (-t, 0, -1), (-t, 0, 1)]
    verts = [np.array(v, dtype=np.float64) / np.linalg.norm(v) for v in verts]
    faces = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6),
             (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10),
             (8, 6, 7), (9, 8, 1)]
    for _ in range(subdivisions):
        cache, new_faces = {}, []

        def mid(i, j):
            key = (min(i, j), max(i, j))
            if key not in cache:
                m = verts[i] + verts[j]
                verts.append(m / np.linalg.norm(m))
                cache[key] = len(verts) - 1
            return cache[key]
        for a, b, c in faces:
            ab, bc, ca = mid(a, b), mid(b, c), mid(c, a)
            new_faces += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        faces = new_faces
    v = np.array(verts) * radius + np.array(center)
    return np.array([[v[a], v[b], v[c]] for a, b, c in faces])


def torus_triangles(n_major=48, n_minor=24, R=1.0, r=0.35, center=(0.0, 0.0, 0.0)):
    """Closed torus (axis z), parametric grid split into triangles; vertices lie ON the analytic torus."""
    u = np.linspace(0.0, 2.0 * np.pi, n_major, endpoint=False)
    v = np.linspace(0.0, 2.0 * np.pi, n_minor, endpoint=False)

    def pt3(i, j):
        a, b = u[i % n_major], v[j % n_minor]
        return np.array([(R + r * np.cos(b)) * np.cos(a), (R + r * np.cos(b)) * np.sin(a), r * np.sin(b)]) + np.array(center)
    tris = []
    for i in range(n_major):
        for j in range(n_minor):
            p00, p10, p11, p01 = pt3(i, j), pt3(i + 1, j), pt3(i + 1, j + 1), pt3(i, j + 1)
            tris.append([p00, p10, p11])
            tris.append([p00, p11, p01])
    return np.array(tris)


def l_extrusion_triangles(height=0.5):
    """L-shaped prism: polygon (0,0)-(2,0)-(2,1)-(1,1)-(1,2)-(0,2) extruded along z in [0, height]; exact planar faces."""
    # caps: a fan over the ring (0,0) (2,0) (2,1) (1,1) (1,2) (0,2) (0,1) -- every cap edge is a ring edge or shared twice
    caps = [[(0, 0), (2, 0), (2, 1)], [(0, 0), (2, 1), (1, 1)], [(0, 0), (1, 1), (0, 1)], [(0, 1), (1, 1), (1, 2)],
            [(0, 1), (1, 2), (0, 2)]]
    tris = []
    for z, flip in ((0.0, True), (height, False)):
        for t in caps:
            pts = [np.array([x, y, z], dtype=np.float64) for x, y in (t[::-1] if flip else t)]
            tris.append(pts)
    # walls over the same ring, so that the surface is watertight
    ring = [(0, 0), (2, 0), (2, 1), (1, 1), (1, 2), (0, 2), (0, 1)]
    for i in range(len(ring)):
        (x0, y0), (x1, y1) = ring[i], ring[(i + 1) % len(ring)]
        a, b = np.array([x0, y0, 0.0]), np.array([x1, y1, 0.0])
        c, d = np.array([x1, y1, height]), np.array([x0, y0, height])
        tris.append([a, b, c])
        tris.append([a, c, d])
    return np.array(tris)


def in_l_extrusion(p, height=0.5, margin=0.0):
    """Analytic classification: +1 inside by more than `margin`, -1 outside by more than `margin`, 0 in the band."""
    x, y, z = p[:, 0], p[:, 1], p[:, 2]

    def box(x0, x1, y0, y1, m):
        return (x > x0 + m) & (x < x1 - m) & (y > y0 + m) & (y < y1 - m) & (z > m) & (z < height - m)
    inside = box(0, 2, 0, 1, margin) | box(0, 1, 0, 2, margin)
    grown = box(0, 2, 0, 1, -margin) | box(0, 1, 0, 2, -margin)
    return np.where(inside, 1, np.where(~grown, -1, 0))


def grid_box_triangles(lo, hi, n=4, flip_every=0):
    """Axis-aligned box whose faces are n x n quads split along one diagonal: many mesh vertices and edges on lattice
    planes. `flip_every` > 0 reverses the winding of every flip_every-th triangle (STL files in the wild are not
    always consistently oriented; the inside test must not care)."""
    lo, hi = np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)
    tris = []
    for axis in range(3):
        u, v = (axis + 1) % 3, (axis + 2) % 3
        for side, x in enumerate((lo[axis], hi[axis])):
            for i in range(n):
                for j in range(n):
                    def corner(a, b):
                        p = np.empty(3)
                        p[axis] = x
                        p[u] = lo[u] + (hi[u] - lo[u]) * a / n
                        p[v] = lo[v] + (hi[v] - lo[v]) * b / n
                        return p
                    q = [corner(i, j), corner(i + 1, j), corner(i + 1, j + 1), corner(i, j + 1)]
                    if side == 0:
                        q = q[::-1]
                    tris.append([q[0], q[1], q[2]])
                    tris.append([q[0], q[2], q[3]])
    tris = np.array(tris)
    if flip_every:
        tris[::flip_every] = tris[::flip_every, ::-1].copy()
    return tris


def ray_through_lattice_points(ext, ys, zs, xs):
    """Points whose +x ray, AFTER the inside test's own y/z nudge (ext * sqrt(2) * 1e-9, ext * sqrt(3) * 1e-9), passes
    exactly through the lattice values ys x zs: undo the nudge in floating point, one ulp at a time."""
    def undo(target, jit):
        p = np.float64(target) - jit
        for _ in range(8):
            s = p + jit
            if s == target:
                return p
            p = np.nextafter(p, np.inf if s < target else -np.inf)
        raise AssertionError("no pre-image")
    jy, jz = np.float64(ext) * 1.4142135623730951e-9, np.float64(ext) * 1.7320508075688772e-9
    return np.array([[x, undo(y, jy), undo(z, jz)] for x in xs for y in ys for z in zs], dtype=np.float64)


def two_box_exact_hit_case(flip_every=0):
    """Two lattice boxes [0,1]^3 and [2,3]x[0,1]^2 in ONE surface, plus points whose nudged +x ray runs exactly through
    mesh vertices, axis-aligned edges and face diagonals. Returns (triangles, points, inside_expected); a ray from the
    first box crosses three faces, from the gap two, from the second box one."""
    tri = np.concatenate([grid_box_triangles((0, 0, 0), (1, 1, 1), 4, flip_every),
                          grid_box_triangles((2, 0, 0), (3, 1, 1), 4, flip_every)])
    ext = 3.0
    lat, gen, xs = [0.25, 0.5, 0.75], [0.1, 0.3721, 0.61], [0.5, 1.5, 2.5]
    sets = [ray_through_lattice_points(ext, lat, lat, xs),          # through vertices
            ray_through_lattice_points(ext, lat, gen, xs),          # through edges of constant y
            ray_through_lattice_points(ext, gen, lat, xs)]          # through edges of constant z
    diag = ray_through_lattice_points(ext, gen, gen, xs)            # through the quad diagonals: nudged y == nudged z
    jy, jz = np.float64(ext) * 1.4142135623730951e-9, np.float64(ext) * 1.7320508075688772e-9
    for r in diag:
        target = r[1] + jy
        z = target - jz
        for _ in range(8):
            s = z + jz
            if s == target:
                break
            z = np.nextafter(z, np.inf if s < target else -np.inf)
        assert z + jz == target
        r[2] = z
    sets.append(diag)
    pts = np.concatenate(sets)
    return tri, pts, (pts[:, 0] == 0.5) | (pts[:, 0] == 2.5)

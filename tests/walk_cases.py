"""Ray queries with closed-form answers for the tree walks (g19_cast_rays): scenes and aimed rays, in FP64, seeded,
no GPU.

An aimed ray is cast at an interior point p of a known primitive from a known distance: origin p - t d, direction d.
Nothing else lies on that segment, so the nearest hit is that primitive at distance t, and an occlusion query
must report a hit below t (1 + eps) and none below t (1 - eps). Unlike a comparison with the oracle on random rays,
every ray has an answer and a single primitive lost by a builder or a walk fails the ray aimed at it.

A case is a dict: "o", "d" (n, 3) FP64; "ids" (n, k) int32, the entity ids any of which is a right answer (-2 pads);
"t" (n,) the expected distance along the unit direction; "normal" (n, 3) the expected normal, facing the ray; "tol"
the allowed |t - expected| (FP32 geometry: a few units in the last place of the coordinates)."""
import math

import numpy as np

DELTA = 1e-3     # distance of the aimed rays' origins (a mesh edge is 0.0226 at n = 708)
MARGIN = 0.05    # least barycentric coordinate of an aimed point
T_TOL = 1e-5     # |t - DELTA| allowed at the heightfield's coordinates (|x| <= 20: an FP32 unit is 1.9e-6 there)


# ---- geometry -------------------------------------------------------------------------------------------------
def quad(a, b, c, d):
    """builtin_scenes.cpp add_quad: the planar quad a-b-c-d as the triangles (a, b, c) and (a, c, d)."""
    return [(a, b, c), (a, c, d)]


def room_triangles():
    """The walls (in push order) and the ceiling light of SCENE_HEIGHTFIELD_ROOM: 14 triangles, entity ids 0-13."""
    x0, x1, y0, y1, z0, z1 = -12.0, 8.0, -8.0, 8.0, -8.0, 8.0
    P = lambda x, y, z: (x, y, z)
    t = []
    t += quad(P(x1, y0, z0), P(x1, y1, z0), P(x1, y1, z1), P(x1, y0, z1))
    t += quad(P(x0, y0, z0), P(x0, y0, z1), P(x0, y1, z1), P(x0, y1, z0))
    t += quad(P(x0, y0, z0), P(x1, y0, z0), P(x1, y1, z0), P(x0, y1, z0))
    t += quad(P(x0, y0, z1), P(x0, y1, z1), P(x1, y1, z1), P(x1, y0, z1))
    t += quad(P(x0, y1, z0), P(x1, y1, z0), P(x1, y1, z1), P(x0, y1, z1))
    t += quad(P(x0, y0, z0), P(x0, y0, z1), P(x1, y0, z1), P(x1, y0, z0))
    zl = z1 - 0.02
    t += quad(P(-5.0, -4.0, zl), P(3.0, -4.0, zl), P(3.0, 4.0, zl), P(-5.0, 4.0, zl))
    return np.array(t, np.float64)


def open_light_triangles():
    """The emitter of the open SCENE_HEIGHTFIELD, pushed after the mesh."""
    return np.array(quad((-14.0, -9.0, -9.0), (-14.0, 9.0, -9.0), (-14.0, 9.0, 9.0), (-14.0, -9.0, 9.0)), np.float64)


def mesh_triangles(n):
    """The heightfield mesh of builtin_scenes.cpp heightfield(), in push order: cell (j, k) (j along y, k along z, k
    outer) gives the triangles 2 (k n + j) and 2 (k n + j) + 1. The vertices are evaluated in the same order of
    operations with the C library's sin and cos, so they equal the engine's bit for bit."""
    g = np.array([-8.0 + 16.0 * float(j) / float(n) for j in range(n + 1)])
    s = np.array([math.sin(0.7 * v) for v in g])
    c = np.array([math.cos(0.9 * v) for v in g])
    x = 6.0 + (1.5 * s)[None, :] * c[:, None]  # [k, j]
    V = np.stack([x, np.broadcast_to(g[None, :], x.shape), np.broadcast_to(g[:, None], x.shape)], -1)
    a, b, cc, d = V[:-1, :-1], V[:-1, 1:], V[1:, 1:], V[1:, :-1]
    tris = np.stack([np.stack([a, b, cc], 2), np.stack([a, cc, d], 2)], 2)  # [k, j, half, vertex, xyz]
    return tris.reshape(-1, 3, 3)


def heightfield_scene(n, room):
    """(triangles (m, 3, 3) in entity order, first mesh entity id) of SCENE_HEIGHTFIELD_ROOM / SCENE_HEIGHTFIELD."""
    mesh = mesh_triangles(n)
    if room:
        return np.concatenate([room_triangles(), mesh]), 14
    return np.concatenate([mesh, open_light_triangles()]), 0


def normals(tris):
    n = np.cross(tris[:, 1] - tris[:, 0], tris[:, 2] - tris[:, 0])
    return n / np.linalg.norm(n, axis=1, keepdims=True)


def interior_points(tris, k, rng):
    """The centroid of every triangle and k - 1 random points with every barycentric coordinate >= MARGIN ->
    (points (m k, 3), triangle index (m k,))."""
    m = len(tris)
    bary = [np.full((m, 3), 1.0 / 3.0)]
    for _ in range(k - 1):
        bary.append(MARGIN + (1.0 - 3.0 * MARGIN) * rng.dirichlet((1.0, 1.0, 1.0), m))
    bary = np.concatenate(bary)
    tri = np.tile(np.arange(m), k)
    return np.einsum("ni,nij->nj", bary, tris[tri]), tri


def unit(d):
    return d / np.linalg.norm(d, axis=1, keepdims=True)


def facing(nrm, d):
    """The normal turned against the ray (the rule of the primary-hit AOV)."""
    return np.where(((nrm * d).sum(1) > 0)[:, None], -nrm, nrm)


def aimed(points, dirs, ids, nrm, t, tol, face=True):
    """Rays ending at `points` after distance t (scalar or per ray) along the unit `dirs`. The expected normal is nrm
    turned against the ray (triangles), or nrm as it is (face=False: a sphere's outward normal)."""
    d = unit(np.asarray(dirs, np.float64).reshape(-1, 3) * np.ones_like(points))
    t = np.broadcast_to(np.asarray(t, np.float64), (len(points),)).copy()
    ids = np.asarray(ids, np.int32)
    ids = ids.reshape(len(points), -1) if ids.ndim > 1 else ids[:, None]
    return {"o": points - t[:, None] * d, "d": d, "ids": ids, "t": t, "normal": facing(nrm, d) if face else nrm, "tol": float(tol)}


def join(*cases):
    k = max(c["ids"].shape[1] for c in cases)
    pad = lambda a: np.pad(a, ((0, 0), (0, k - a.shape[1])), constant_values=-2)
    out = {key: np.concatenate([c[key] for c in cases]) for key in ("o", "d", "t", "normal")}
    out["ids"] = np.concatenate([pad(c["ids"]) for c in cases])
    out["tol"] = max(c["tol"] for c in cases)
    return out


def subset(case, idx):
    out = {k: v[idx] for k, v in case.items() if k != "tol"}
    out["tol"] = case["tol"]
    return out


def occlusion_pairs(case):
    """The occlusion queries of an aimed case: tmax = t + 2 tol must report a hit, tmax = t - 2 tol must not (the
    bracket is twice the allowed FP32 error of t: 1e-3 (1 +- 2e-2) on the heightfield)."""
    return case["t"] + 2 * case["tol"], case["t"] - 2 * case["tol"]


# ---- the heightfield scenes at full size -------------------------------------------------------------------
def heightfield_cases(n, room, points_per_tri=2, wall_points=256, seed=0):
    """The aimed sets of SCENE_HEIGHTFIELD(_ROOM) with n x n cells:
    "axis": every mesh triangle, rays along +x and -x (the surface is a function of (y, z): the line meets it once);
    "normal": every mesh triangle, rays along -n from p + DELTA n;
    "walls": the room's walls and light (or the open scene's emitter), big primitives and merged parallelograms, both
    halves, rays along -n and +n. A wall ray from inside the room is kept only where it cannot meet the mesh's rim,
    which touches the side walls, floor and ceiling at x in [4.5, 7.5]."""
    rng = np.random.default_rng(seed)
    tris, first = heightfield_scene(n, room)
    nrm = normals(tris)
    m = 2 * n * n
    mesh = np.arange(first, first + m)
    p, k = interior_points(tris[mesh], points_per_tri, rng)
    ids, nk = mesh[k], nrm[mesh][k]
    ex = np.array([1.0, 0.0, 0.0])
    axis = join(aimed(p, ex, ids, nk, DELTA, T_TOL), aimed(p, -ex, ids, nk, DELTA, T_TOL))
    normal = aimed(p, -nk, ids, nk, DELTA, T_TOL)
    other = np.setdiff1d(np.arange(len(tris)), mesh)
    wp, wk = interior_points(tris[other], wall_points, rng)
    wids, wn = other[wk], nrm[other][wk]
    sides = [aimed(wp, -wn, wids, wn, DELTA, T_TOL), aimed(wp, wn, wids, wn, DELTA, T_TOL)]
    if room:
        for i, c in enumerate(sides):
            inside = ((c["o"] > ROOM_LO) & (c["o"] < ROOM_HI)).all(1)
            sides[i] = subset(c, ~(inside & (wp[:, 0] >= 4.4) & (wp[:, 0] <= 7.6)))
    return {"axis": axis, "normal": normal, "walls": join(*sides)}


ROOM_LO, ROOM_HI = np.array([-12.0, -8.0, -8.0]), np.array([8.0, 8.0, 8.0])


def closed_room_rays(count, seed=0):
    """count rays from uniform points inside the room, in uniform directions (FP64), and for each whether its exit
    from the room box lies within 1e-5 of a box edge, where two walls' parallelograms meet and FP32 intersection is
    not watertight: the only rays allowed to miss."""
    rng = np.random.default_rng(seed)
    o = rng.uniform(ROOM_LO + 1e-3, ROOM_HI - 1e-3, (count, 3))
    d = unit(rng.normal(size=(count, 3)))
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(d > 0, (ROOM_HI - o) / d, np.where(d < 0, (ROOM_LO - o) / d, np.inf)).min(1)
    q = o + t[:, None] * d
    on = (np.abs(q - ROOM_LO) <= 1e-5) | (np.abs(q - ROOM_HI) <= 1e-5)
    return o, d, on.sum(1) >= 2


# ---- direction variants ----------------------------------------------------------------------------------------
def axis_variants(case):
    """Copies of an axis-aligned case whose zero direction components are -0.0, 1e-30 and 1e-38 (below FP32's
    normal range: flushed to zero by the kernels) instead of +0.0. The answers must not change."""
    out = []
    zero = case["d"] == 0
    for v in (-0.0, 1e-30, -1e-30, 1e-38):
        c = dict(case)
        c["d"] = np.where(zero, v, case["d"])
        out.append(c)
    return out


# ---- builder edge cases ----------------------------------------------------------------------------------------
# An edge case: {"root": (lo, hi) of the Octree, "prims": [("tri", v0, v1, v2) | ("sph", centre, radius)] in entity
# order, "cases": {name: aimed case}}.

def _tri_cases(tris, ids, rng, dirs, t, tol, k=2):
    """Aimed rays at k interior points of each triangle along each of `dirs` (an (3,) direction, or "n" for -n)."""
    nrm = normals(tris)
    p, j = interior_points(tris, k, rng)
    ids = np.asarray(ids)[j]
    parts = []
    for d in dirs:
        dd = -nrm[j] if isinstance(d, str) else np.asarray(d, np.float64)
        parts.append(aimed(p, dd, ids, nrm[j], t, tol))
    return join(*parts)


def _fp32_tol(extent):
    """32 FP32 units at the scene's largest coordinate, at least T_TOL."""
    return max(T_TOL, 32.0 * float(np.spacing(np.float32(extent))))


def _surface(n, lo, hi, x0, amp):
    """A curved n x n patch x = x0 + amp sin(y) cos(z) over [lo, hi]^2 (a mesh no two of whose triangles merge)."""
    g = np.linspace(lo, hi, n + 1)
    x = x0 + amp * np.sin(g)[None, :] * np.cos(g)[:, None]
    V = np.stack([x, np.broadcast_to(g[None, :], x.shape), np.broadcast_to(g[:, None], x.shape)], -1)
    a, b, c, d = V[:-1, :-1], V[:-1, 1:], V[1:, 1:], V[1:, :-1]
    return np.stack([np.stack([a, b, c], 2), np.stack([a, c, d], 2)], 2).reshape(-1, 3, 3)


def case_duplicates(seed=1):
    """Every triangle of a curved patch pushed 2-5 times in a row: equal boxes, equal Morton codes, split by position
    only. Any of the copies is a right answer."""
    rng = np.random.default_rng(seed)
    tris = _surface(12, -2.0, 2.0, 1.0, 0.3)
    reps = rng.integers(2, 6, len(tris))
    prims, groups = [], []
    for tr, r in zip(tris, reps):
        groups.append(list(range(len(prims), len(prims) + r)) + [-2] * (5 - r))
        prims += [("tri",) + tuple(tr)] * r
    ex = np.array([1.0, 0.0, 0.0])
    c = _tri_cases(tris, np.arange(len(tris)), rng, (ex, -ex, "n"), DELTA, T_TOL)
    return {"root": ((-20,) * 3, (20,) * 3), "prims": prims,
            "cases": {"dup": dict(c, ids=np.array(groups, np.int32)[c["ids"][:, 0]])}}


def _lattice_triangle(cell, size, rng):
    """A triangle of extent `size` in the plane x = const through the centre of a 4-unit lattice cell, tilted a little."""
    c = np.array(cell, np.float64) * 4.0
    u = np.array([0.1, 1.0, 0.0]) * size / 2
    v = np.array([0.05, 0.0, 1.0]) * size / 2
    return np.array([c - u - v, c + u - v, c + v * rng.uniform(0.8, 1.0)])


def case_bvh_sizes(n_small, n_big, seed=2):
    """n_big triangles larger than 1/32 of the root box (the first 64, largest first, are kept out of the hierarchy and
    tested first; the rest go in) and n_small small ones, each alone in a 4-unit lattice cell. With 12 big triangles
    the hierarchy holds exactly n_small primitives: a single leaf while n_small <= bvh_leaf, a node above that."""
    rng = np.random.default_rng(seed + 100 * n_small + n_big)
    cells = [(i, j, k) for i in range(-4, 5) for j in range(-4, 5) for k in range(-4, 5)]
    order = rng.permutation(len(cells))
    tris = [_lattice_triangle(cells[order[i]], 1.4 + 1.5 * i / max(1, n_big), rng) for i in range(n_big)]
    tris += [_lattice_triangle(cells[order[n_big + i]], rng.uniform(0.1, 0.5), rng) for i in range(n_small)]
    tris = np.array(tris)
    ex = np.array([1.0, 0.0, 0.0])
    c = _tri_cases(tris, np.arange(len(tris)), rng, (ex, -ex, "n"), DELTA, T_TOL, k=8)
    return {"root": ((-20,) * 3, (20,) * 3), "prims": [("tri",) + tuple(t) for t in tris], "cases": {"aimed": c}}


def case_root_faces(seed=3):
    """Small triangles with a vertex on each of the six faces of the root box [-1, 1]^3 and at its eight corners (their
    quantised boxes clamp at 0 and 65535; the Octree rejects an entity that only touches its box, so the other
    vertices lean inwards), and a strip of triangles smaller than one quantisation step (2 / 65535), side by side.
    Rays come at the face triangles from inside and from outside the root box."""
    rng = np.random.default_rng(seed)
    tris = []
    s = 0.05  # below 1/32 of the root: inside the hierarchy
    for axis in range(3):
        for sign in (-1.0, 1.0):
            for off in ((0.3, -0.2), (-0.5, 0.6)):
                a, b = [k for k in range(3) if k != axis]
                v0 = np.zeros(3)
                v0[axis], v0[a], v0[b] = sign, off[0], off[1]
                v1, v2 = v0.copy(), v0.copy()
                v1[a] += s
                v2[b] += s
                v1[axis] -= 0.2 * s * sign
                v2[axis] -= 0.2 * s * sign
                tris.append([v0, v1, v2])
    for cx in (-1.0, 1.0):
        for cy in (-1.0, 1.0):
            for cz in (-1.0, 1.0):
                c = np.array([cx, cy, cz])
                tris.append([c, c - s * np.array([0.2 * cx, cy, 0.2 * cz]), c - s * np.array([0.2 * cx, 0.2 * cy, cz])])
    h = 1.5e-5
    for i in range(16):
        y0, z0 = 0.1 + i * h, 0.2
        tris.append([np.array([0.3, y0, z0]), np.array([0.3, y0 + h, z0]), np.array([0.3, y0, z0 + h])])
    tris = np.array(tris)
    nrm = normals(tris)
    p, j = interior_points(tris, 4, rng)
    ids, nj = np.arange(len(tris))[j], nrm[j]
    c = join(aimed(p, nj, ids, nj, DELTA, T_TOL), aimed(p, -nj, ids, nj, DELTA, T_TOL))
    return {"root": ((-1,) * 3, (1,) * 3), "prims": [("tri",) + tuple(t) for t in tris], "cases": {"aimed": c}}


def plane_triangles(count):
    """The first `count` triangles of a 64 x 64-cell plane at z = 0.5 over [-4, 4]^2: every cell's lower triangle, then
    every upper one (no two consecutive triangles share an edge, so none merge into a parallelogram)."""
    g = np.linspace(-4.0, 4.0, 65)
    Y, X = np.meshgrid(g, g, indexing="ij")
    V = np.stack([X, Y, np.full_like(X, 0.5)], -1)
    a, b, c, d = V[:-1, :-1], V[:-1, 1:], V[1:, 1:], V[1:, :-1]
    lower = np.stack([a, b, c], 2).reshape(-1, 3, 3)
    upper = np.stack([a, c, d], 2).reshape(-1, 3, 3)
    return np.concatenate([lower, upper])[:count]


def case_plane(count, seed=4):
    """A plane of `count` triangles at one z: every box is flat in z. 4096 primitives is where the octree is built on
    the device instead of the host. Axis rays along +-z and oblique rays from both sides."""
    rng = np.random.default_rng(seed + count)
    tris = plane_triangles(count)
    ez = np.array([0.0, 0.0, 1.0])
    dirs = (ez, -ez, unit(np.array([[0.3, -0.2, 1.0]]))[0], unit(np.array([[-0.4, 0.25, -1.0]]))[0])
    c = _tri_cases(tris, np.arange(len(tris)), rng, dirs, DELTA, T_TOL, k=1)
    return {"root": ((-20,) * 3, (20,) * 3), "prims": [("tri",) + tuple(t) for t in tris],
            "cases": {"axis": subset(c, slice(0, 2 * count)), "oblique": subset(c, slice(2 * count, None))}}


def case_translated(offset, seed=5):
    """A curved patch moved by (offset, -offset, offset): the slab offsets (root_lo - o) / d are differences of large
    numbers there. The tolerance and the distance grow with the FP32 unit. (No spheres: an ImpSphere's Octree box is
    centred on the origin, as in the reference, so the Octree rejects one far from it.)"""
    rng = np.random.default_rng(seed)
    T = np.array([offset, -offset, offset], np.float64)
    tris = _surface(6, -1.0, 1.0, 0.0, 0.3) + T
    tol = _fp32_tol(2.0 * offset)
    delta = max(DELTA, 8 * tol)
    ex = np.array([1.0, 0.0, 0.0])
    c = _tri_cases(tris, np.arange(len(tris)), rng, (ex, -ex, "n"), delta, tol)
    return {"root": (tuple(T - 20), tuple(T + 20)), "prims": [("tri",) + tuple(t) for t in tris], "cases": {"aimed": c}}


def case_spheres(seed=6):
    """Small spheres on a grid at z = 0 with small upright triangles between them, so that leaves hold both kinds.
    Spheres: rays at the centre along -z from 2 above (t = 2 - r), and from the centre outwards in random directions
    (t = r; a sphere's normal is the outward one either way). Triangles: axis rays along +-x and oblique ones."""
    rng = np.random.default_rng(seed)
    cen, rad, tris = [], [], []
    for i in range(6):
        for j in range(6):
            cen.append((float(i), float(j), 0.0))
            rad.append(rng.uniform(0.1, 0.3))
            y, z = float(j) + rng.uniform(-0.1, 0.1), rng.uniform(-0.1, 0.1)
            tris.append([(i + 0.5, y - 0.1, z - 0.1), (i + 0.5, y + 0.1, z - 0.1), (i + 0.5, y, z + 0.1)])
    cen, rad, tris = np.array(cen), np.array(rad), np.array(tris)
    prims, sph_ids, tri_ids = [], [], []
    for k in range(len(cen)):  # interleaved in entity order too
        sph_ids.append(len(prims))
        prims.append(("sph", cen[k], rad[k]))
        tri_ids.append(len(prims))
        prims.append(("tri",) + tuple(tris[k]))
    sph_ids = np.array(sph_ids)
    ez = np.array([0.0, 0.0, 1.0])
    top = cen + rad[:, None] * ez
    above = aimed(top, -ez, sph_ids, np.tile(ez, (len(cen), 1)), 2.0 - rad, T_TOL)
    u = unit(rng.normal(size=(4 * len(cen), 3)))
    k = np.repeat(np.arange(len(cen)), 4)
    inside = aimed(cen[k] + rad[k, None] * u, u, sph_ids[k], u, rad[k], T_TOL, face=False)
    ex = np.array([1.0, 0.0, 0.0])
    t = _tri_cases(tris, np.array(tri_ids), rng, (ex, -ex, unit(np.array([[1.0, 0.3, -0.2]]))[0]), DELTA, T_TOL)
    return {"root": ((-20,) * 3, (20,) * 3), "prims": prims, "cases": {"spheres": join(above, inside), "triangles": t}}


def edge_cases():
    """name -> edge case (built on demand: the plane cases hold up to 8192 triangles)."""
    cases = {"duplicates": case_duplicates}
    for b in (1, 2, 4, 5, 8, 9):
        cases["bvh_%d_small" % b] = lambda b=b: case_bvh_sizes(b, 12)
    cases["bvh_all_big"] = lambda: case_bvh_sizes(0, 20)
    cases["bvh_72_big"] = lambda: case_bvh_sizes(3, 72)
    cases["root_faces"] = case_root_faces
    for n in (4095, 4096, 4097, 8192):
        cases["plane_%d" % n] = lambda n=n: case_plane(n)
    cases["translated_1e3"] = lambda: case_translated(1e3)
    cases["translated_1e4"] = lambda: case_translated(1e4)
    cases["spheres"] = case_spheres
    return cases


def build_octree(g19, case):
    """The edge case as an Octree of ImpTriangles and ImpSpheres, in entity order."""
    lo, hi = case["root"]
    sc = g19.Octree(tuple(float(v) for v in lo), tuple(float(v) for v in hi))
    for p in case["prims"]:
        if p[0] == "tri":
            idx, ok = sc.push_back(g19.ImpTriangle(tuple(p[1]), tuple(p[2]), tuple(p[3]), (0.7, 0.7, 0.7)))
        else:
            idx, ok = sc.push_back(g19.ImpSphere(tuple(p[1]), float(p[2]), (0.7, 0.7, 0.7)))
        assert ok, "entity %d rejected by the Octree" % idx
    return sc

"""Seeded procedural scenes for the BDPT core (BASELINE.json configs 1, 2, 4, 5).

The reference's own scenes are absent git-LFS blobs (SURVEY.md section 2 row 13: Content/**), so
every scene here is generated: shoebox (12 triangles, 6 materials), furnished room (~100 k),
mine tunnels (~1 M), concert hall (~5 M).  Triangles are float32 [T][3][3] in metres; each
triangle carries a material id into an [M][B] absorption table -- the build's equivalent of
UAcousticGeometryComponent -> UAcousticMaterial::Absorption (GEO.h:9-22, MAT.h:16-34).

No wall-clock, no global RNG: everything derives from numpy Generator(PCG64(seed)).
"""
import numpy as np

# 8 octave bands 63 Hz .. 8 kHz.  Names follow Content/StarterContent/AudioMaterials/MAT_*.
MATERIAL_NAMES = ["concrete", "wood", "glass", "carpet", "curtain", "seat", "plaster", "metal"]
MATERIAL_ABSORPTION = np.array([
    [0.01, 0.01, 0.02, 0.02, 0.02, 0.03, 0.04, 0.05],   # concrete
    [0.15, 0.11, 0.10, 0.07, 0.06, 0.07, 0.08, 0.09],   # wood
    [0.35, 0.25, 0.18, 0.12, 0.07, 0.04, 0.03, 0.02],   # glass
    [0.02, 0.06, 0.14, 0.37, 0.60, 0.65, 0.65, 0.70],   # carpet
    [0.07, 0.31, 0.49, 0.75, 0.70, 0.60, 0.55, 0.50],   # curtain
    [0.40, 0.50, 0.58, 0.61, 0.58, 0.50, 0.45, 0.40],   # seat
    [0.14, 0.10, 0.06, 0.05, 0.04, 0.03, 0.03, 0.03],   # plaster
    [0.04, 0.04, 0.03, 0.03, 0.02, 0.02, 0.02, 0.02],   # metal
], dtype=np.float32)


def absorption_table(n_bands=8, n_mats=8):
    """[n_mats][n_bands] absorption; n_bands < 8 takes the centre bands (B=1 -> the 1 kHz band,
    the analogue of the reference's single Absorption[2] read, SUB.cpp:385)."""
    lo = (8 - n_bands) // 2
    return np.ascontiguousarray(MATERIAL_ABSORPTION[:n_mats, lo:lo + n_bands])


class Scene:
    def __init__(self, name, verts, tri_mat, absorption, sources, listener, meta=None):
        self.name = name
        self.verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
        self.tri_mat = np.ascontiguousarray(tri_mat, dtype=np.uint32)
        self.absorption = np.ascontiguousarray(absorption, dtype=np.float32)
        self.sources = np.ascontiguousarray(sources, dtype=np.float32).reshape(-1, 3)
        self.listener = np.ascontiguousarray(listener, dtype=np.float32).reshape(3)
        self.meta = meta or {}
        assert len(self.verts) == len(self.tri_mat)

    @property
    def n_tris(self):
        return len(self.verts)


# ---------------------------------------------------------------------------------------------
# primitives (all return float32 [n][3][3])
# ---------------------------------------------------------------------------------------------
def _grid_tris(P):
    """P: [nu+1][nv+1][3] vertex grid -> 2*nu*nv triangles sharing the grid vertices"""
    a = P[:-1, :-1]
    b = P[1:, :-1]
    c = P[1:, 1:]
    d = P[:-1, 1:]
    t1 = np.stack([a, b, c], axis=-2)
    t2 = np.stack([a, c, d], axis=-2)
    return np.concatenate([t1.reshape(-1, 3, 3), t2.reshape(-1, 3, 3)], axis=0).astype(np.float32)


def patch(origin, du, dv, nu=1, nv=1):
    origin, du, dv = (np.asarray(x, dtype=np.float64) for x in (origin, du, dv))
    u = np.linspace(0.0, 1.0, nu + 1)[:, None, None]
    v = np.linspace(0.0, 1.0, nv + 1)[None, :, None]
    return _grid_tris(origin + u * du + v * dv)


def box(lo, hi, tess=1):
    """6 faces, each tess x tess quads; returns (tris, face_id[ntris]) with face order
    -x, +x, -y, +y, -z (floor), +z (ceiling)"""
    lo = np.asarray(lo, dtype=np.float64)
    hi = np.asarray(hi, dtype=np.float64)
    s = hi - lo
    ex, ey, ez = np.array([s[0], 0, 0]), np.array([0, s[1], 0]), np.array([0, 0, s[2]])
    faces = [
        patch(lo, ey, ez, tess, tess), patch(lo + ex, ey, ez, tess, tess),
        patch(lo, ex, ez, tess, tess), patch(lo + ey, ex, ez, tess, tess),
        patch(lo, ex, ey, tess, tess), patch(lo + ez, ex, ey, tess, tess),
    ]
    ids = np.concatenate([np.full(len(f), i, dtype=np.uint32) for i, f in enumerate(faces)])
    return np.concatenate(faces, axis=0), ids


def uv_sphere(center, radius, n_lat, n_lon, squash=(1.0, 1.0, 1.0)):
    th = np.linspace(0.0, np.pi, n_lat + 1)[:, None]
    ph = np.linspace(0.0, 2.0 * np.pi, n_lon + 1)[None, :]
    ph = np.where(np.arange(n_lon + 1)[None, :] == n_lon, 0.0, ph)    # close the seam exactly
    x = np.sin(th) * np.cos(ph)
    y = np.sin(th) * np.sin(ph)
    z = np.cos(th) * np.ones_like(ph)
    P = np.stack([x, y, z], axis=-1) * radius * np.asarray(squash) + np.asarray(center, dtype=np.float64)
    return _grid_tris(P)


def tube(path, radii_fn, n_ring, seed_noise=None, noise_amp=0.0):
    """Closed tube along polyline `path` [n][3]; ring vertices displaced by seeded noise.
    Returns triangles incl. end caps (watertight: caps reuse the end ring vertices)."""
    path = np.asarray(path, dtype=np.float64)
    n = len(path)
    tang = np.gradient(path, axis=0)
    tang /= np.linalg.norm(tang, axis=1, keepdims=True)
    up = np.array([0.0, 0.0, 1.0])
    side = np.cross(tang, up)
    side /= np.maximum(np.linalg.norm(side, axis=1, keepdims=True), 1e-9)
    up2 = np.cross(side, tang)
    ang = np.linspace(0.0, 2.0 * np.pi, n_ring + 1)
    ang[-1] = 0.0
    r = radii_fn(n, n_ring + 1)
    if seed_noise is not None and noise_amp > 0:
        rng = np.random.Generator(np.random.PCG64(seed_noise))
        nz = rng.uniform(-noise_amp, noise_amp, size=(n, n_ring))
        nz = np.concatenate([nz, nz[:, :1]], axis=1)
        r = r + nz
    ca, sa = np.cos(ang)[None, :, None], np.sin(ang)[None, :, None]
    P = path[:, None, :] + r[:, :, None] * (ca * side[:, None, :] + sa * up2[:, None, :])
    tris = [_grid_tris(P)]
    for end, c in ((0, path[0]), (n - 1, path[-1])):
        ring = P[end]
        cap = np.stack([np.broadcast_to(c, ring[:-1].shape), ring[:-1], ring[1:]], axis=1)
        tris.append(cap.astype(np.float32))
    return np.concatenate(tris, axis=0)


# ---------------------------------------------------------------------------------------------
# config 1: shoebox
# ---------------------------------------------------------------------------------------------
def shoebox(size=(7.0, 5.0, 3.0), n_bands=8):
    """12 triangles, 6 materials (one per wall).  Source (1.5,1.2,1.0), listener (5.0,3.5,1.6)
    per SURVEY.md section 8d config 1."""
    tris, face = box((0, 0, 0), size, 1)
    mats = np.array([0, 6, 2, 1, 3, 4], dtype=np.uint32)[face]    # walls..., carpet floor, curtain ceiling
    return Scene("shoebox", tris, mats, absorption_table(n_bands),
                 [[1.5, 1.2, 1.0]], [5.0, 3.5, 1.6], {"size": size})


# ---------------------------------------------------------------------------------------------
# config 2: furnished room
# ---------------------------------------------------------------------------------------------
def furnished_room(seed=1, target_tris=100_000, n_bands=8, size=(12.0, 9.0, 3.6)):
    rng = np.random.Generator(np.random.PCG64(seed))
    size = np.asarray(size, dtype=np.float64)
    src = np.array([2.0, 1.8, 1.4])
    lis = np.array([9.5, 6.5, 1.6])
    parts, mats = [], []

    def add(t, m):
        parts.append(t)
        mats.append(np.full(len(t), m, dtype=np.uint32) if np.isscalar(m) else m)

    wall_tess = 24
    t, face = box((0, 0, 0), size, wall_tess)
    add(t, np.array([6, 6, 2, 6, 3, 6], dtype=np.uint32)[face])
    budget = target_tris - len(t)

    def clear(c, r):
        return min(np.linalg.norm(c - src), np.linalg.norm(c - lis)) > r + 0.6

    # tables: top slab + 4 legs (wood), cabinets (boxes, wood/metal), upholstered blobs (seat)
    n_sph_lat, n_sph_lon = 20, 40
    sph_tris = 2 * n_sph_lat * n_sph_lon
    box_tess = 3
    box_tris = 12 * box_tess * box_tess
    n_sph = int(0.55 * budget / sph_tris)
    n_box = int(0.45 * budget / (box_tris * 1.72))
    placed = 0
    while placed < n_sph:
        r = rng.uniform(0.18, 0.45)
        c = np.array([rng.uniform(r + 0.1, size[0] - r - 0.1), rng.uniform(r + 0.1, size[1] - r - 0.1),
                      rng.uniform(r, 1.4)])
        sq = (1.0, 1.0, rng.uniform(0.6, 1.0))
        if not clear(c, r):
            continue
        add(uv_sphere(c, r, n_sph_lat, n_sph_lon, sq), int(rng.choice([5, 4, 3])))
        placed += 1
    placed = 0
    while placed < n_box:
        w = rng.uniform(0.4, 1.6, size=2)
        h = rng.uniform(0.4, 2.2)
        c = np.array([rng.uniform(w[0], size[0] - w[0]), rng.uniform(w[1], size[1] - w[1]), 0.0])
        if not clear(c + [0, 0, h / 2], max(w.max(), h) * 0.75):
            continue
        lo = c - [w[0] / 2, w[1] / 2, 0]
        if rng.uniform() < 0.5:      # cabinet
            add(box(lo + [0, 0, 0.02], lo + [w[0], w[1], h], box_tess)[0], int(rng.choice([1, 7])))
            add(box(lo + [0.05, 0.05, h], lo + [w[0] - 0.05, w[1] - 0.05, h + 0.04], box_tess)[0], 1)
        else:                        # table: slab + 4 legs
            ht = rng.uniform(0.6, 0.9)
            add(box(lo + [0, 0, ht], lo + [w[0], w[1], ht + 0.05], box_tess)[0], 1)
            for sx in (0.05, w[0] - 0.11):
                for sy in (0.05, w[1] - 0.11):
                    add(box(lo + [sx, sy, 0.02], lo + [sx + 0.06, sy + 0.06, ht], 1)[0], 7)
        placed += 1
    verts = np.concatenate(parts, axis=0)
    tri_mat = np.concatenate(mats)
    return Scene("furnished_room", verts, tri_mat, absorption_table(n_bands), [src], lis,
                 {"size": tuple(size), "seed": seed})


# ---------------------------------------------------------------------------------------------
# config 4: mine tunnels
# ---------------------------------------------------------------------------------------------
def mine_tunnels(seed=4, target_tris=1_000_000, n_sources=64, n_bands=8):
    rng = np.random.Generator(np.random.PCG64(seed))
    n_ring = 96
    n_seg = max(8, int(target_tris * 0.9 / (2 * n_ring)))
    # meandering centre line, 0.25 m steps
    step = 0.25
    heading = np.cumsum(rng.normal(0.0, 0.02, size=n_seg))
    pitch = 0.05 * np.sin(np.linspace(0, 6 * np.pi, n_seg))
    d = np.stack([np.cos(heading) * np.cos(pitch), np.sin(heading) * np.cos(pitch), np.sin(pitch)], axis=1)
    path = np.cumsum(d * step, axis=0)

    def radii(n, m):
        base = 1.6 + 0.35 * np.sin(np.linspace(0, 40 * np.pi, n))[:, None]
        ang = np.linspace(0, 2 * np.pi, m)[None, :]
        return base * (1.0 - 0.25 * (np.sin(ang) < -0.6))          # flattened floor

    t = tube(path, radii, n_ring, seed_noise=seed + 1, noise_amp=0.08)
    parts = [t]
    mats = [np.zeros(len(t), dtype=np.uint32)]
    # props: support beams (boxes) every few metres
    remaining = target_tris - len(t)
    n_props = max(0, remaining // 12)
    idx = np.linspace(10, n_seg - 10, n_props).astype(int) if n_props else []
    for k, i in enumerate(idx):
        c = path[i]
        off = np.array([rng.uniform(-0.9, 0.9), rng.uniform(-0.9, 0.9), -0.6])
        s = rng.uniform(0.05, 0.25, size=3)
        parts.append(box(c + off - s, c + off + s, 1)[0])
        mats.append(np.full(12, 1 if k % 2 else 7, dtype=np.uint32))
    verts = np.concatenate(parts, axis=0)
    tri_mat = np.concatenate(mats)
    sidx = np.linspace(20, n_seg - 20, n_sources).astype(int)
    sources = path[sidx] + [0, 0, 0.3]
    listener = path[n_seg // 2] + [0, 0, 0.4]
    return Scene("mine_tunnels", verts, tri_mat, absorption_table(n_bands), sources, listener,
                 {"seed": seed, "length_m": float(n_seg * step)})


# ---------------------------------------------------------------------------------------------
# config 5: concert hall
# ---------------------------------------------------------------------------------------------
def concert_hall(seed=5, target_tris=5_000_000, n_bands=8):
    rng = np.random.Generator(np.random.PCG64(seed))
    size = np.array([48.0, 30.0, 18.0])
    parts, mats = [], []

    def add(t, m):
        parts.append(t)
        mats.append(np.full(len(t), m, dtype=np.uint32) if np.isscalar(m) else m)

    scale = (target_tris / 5_000_000.0) ** 0.5
    wall_tess = max(4, int(160 * scale))
    t, face = box((0, 0, 0), size, wall_tess)
    add(t, np.array([6, 6, 1, 1, 3, 6], dtype=np.uint32)[face])
    # stage
    add(box((2, 6, 0.01), (12, 24, 1.2), max(2, int(24 * scale)))[0], 1)
    # tiered seating: rows of seats, each seat a squashed sphere + back box
    n_lat, n_lon = 10, 16
    seat_tris = 2 * n_lat * n_lon + 12
    used = sum(len(p) for p in parts)
    n_diff = int(0.15 * (target_tris - used) / (2 * 6 * 6))
    n_seats = int(0.85 * (target_tris - used) / seat_tris)
    rows = max(1, int(np.sqrt(n_seats / 1.6)))
    cols = max(1, n_seats // rows)
    xs = np.linspace(15.0, 45.0, rows)
    ys = np.linspace(2.0, 28.0, cols)
    unit = uv_sphere((0, 0, 0), 1.0, n_lat, n_lon).astype(np.float64)
    backb = box((-0.5, -0.5, -0.5), (0.5, 0.5, 0.5), 1)[0].astype(np.float64)
    rise = 0.12
    pitch_x = (xs[1] - xs[0]) if rows > 1 else 1.0
    pitch_y = (ys[1] - ys[0]) if cols > 1 else 1.0
    sx, sy = 0.42 * min(pitch_x, 0.9), 0.42 * min(pitch_y, 0.6)
    cx, cy = np.meshgrid(xs, ys, indexing="ij")
    cz = 0.45 + rise * (cx - 15.0)
    centres = np.stack([cx, cy, cz], axis=-1).reshape(-1, 1, 1, 3)
    jitter = rng.uniform(-0.01, 0.01, size=centres.shape)
    seats = unit[None] * np.array([sx, sy, 0.18]) + centres + jitter
    add(seats.reshape(-1, 3, 3).astype(np.float32), 5)
    backs = backb[None] * np.array([0.08, 2 * sy, 0.5]) + centres + [sx, 0, 0.3]
    add(backs.reshape(-1, 3, 3).astype(np.float32), 5)
    # diffuser panels on side walls / ceiling
    for k in range(n_diff):
        w = rng.uniform(0.4, 1.5)
        if k % 3 == 0:
            o = np.array([rng.uniform(1, 46), 0.05 + rng.uniform(0, 0.3), rng.uniform(3, 16)])
            add(patch(o, [w, rng.uniform(-0.2, 0.2), 0], [0, rng.uniform(-0.2, 0.2), w], 6, 6), 1)
        elif k % 3 == 1:
            o = np.array([rng.uniform(1, 46), 29.95 - rng.uniform(0, 0.3), rng.uniform(3, 16)])
            add(patch(o, [w, rng.uniform(-0.2, 0.2), 0], [0, rng.uniform(-0.2, 0.2), w], 6, 6), 1)
        else:
            o = np.array([rng.uniform(1, 46), rng.uniform(1, 28), 17.9 - rng.uniform(0, 0.5)])
            add(patch(o, [w, 0, rng.uniform(-0.2, 0.2)], [0, w, rng.uniform(-0.2, 0.2)], 6, 6), 6)
    verts = np.concatenate(parts, axis=0)
    tri_mat = np.concatenate(mats)
    return Scene("concert_hall", verts, tri_mat, absorption_table(n_bands),
                 [[7.0, 15.0, 2.8]], [30.0, 14.0, 0.45 + rise * 15.0 + 1.2],
                 {"seed": seed, "size": tuple(size)})


# ---------------------------------------------------------------------------------------------
# moving geometry: two rooms joined by a doorway with a hinged door
# ---------------------------------------------------------------------------------------------
def door_rooms(seed=11, n_bands=8, wall_tess=16, n_blobs=4):
    """Two 6 x 8 x 3 m rooms side by side (x < 6 and x > 6.2), a 0.2 m dividing wall with a 1.0 x 2.1 m doorway at
    y = 3.5 .. 4.5, and a 4 cm wooden door hinged on the vertical line (6.1, 3.5).  The source is in the first room, the
    listener in the second; each room holds a few upholstered blobs and cabinets.  meta["door"] = (first triangle, count)
    of the door, the last part of the scene; door_verts() swings it.  Surfaces are opaque (no transmission by default), so
    with the door closed no path connects the two rooms and the listener's histogram is empty."""
    rng = np.random.Generator(np.random.PCG64(seed))
    X0, W, X1, Y, Z = 6.0, 0.2, 12.2, 8.0, 3.0
    y0, y1, zd = 3.5, 4.5, 2.1
    src = np.array([2.0, 2.0, 1.4])
    lis = np.array([10.0, 6.0, 1.6])
    parts, mats = [], []

    def add(t, m):
        parts.append(t)
        mats.append(np.full(len(t), m, dtype=np.uint32) if np.isscalar(m) else m)

    t, face = box((0, 0, 0), (X1, Y, Z), wall_tess)
    add(t, np.array([6, 6, 2, 6, 3, 6], dtype=np.uint32)[face])
    for x in (X0, X0 + W):                                          # the two faces of the dividing wall around the doorway
        add(patch([x, 0, 0], [0, y0, 0], [0, 0, Z], 6, 6), 6)
        add(patch([x, y1, 0], [0, Y - y1, 0], [0, 0, Z], 6, 6), 6)
        add(patch([x, y0, zd], [0, y1 - y0, 0], [0, 0, Z - zd], 2, 2), 6)
    add(patch([X0, y0, 0], [W, 0, 0], [0, 0, zd], 2, 6), 6)        # jambs and lintel
    add(patch([X0, y1, 0], [W, 0, 0], [0, 0, zd], 2, 6), 6)
    add(patch([X0, y0, zd], [W, 0, 0], [0, y1 - y0, 0], 2, 2), 6)
    for lo_x, hi_x in ((0.0, X0), (X0 + W, X1)):                   # furniture, clear of the source, listener and door swing
        placed = 0
        while placed < n_blobs:
            r = rng.uniform(0.25, 0.5)
            c = np.array([rng.uniform(lo_x + r + 0.1, hi_x - r - 0.1), rng.uniform(r + 0.1, Y - r - 0.1), rng.uniform(r, 1.2)])
            if min(np.linalg.norm(c - src), np.linalg.norm(c - lis), np.linalg.norm(c[:2] - [X0 + W / 2, 4.0])) < r + 1.4:
                continue
            add(uv_sphere(c, r, 20, 40, (1.0, 1.0, rng.uniform(0.6, 1.0))), int(rng.choice([5, 4, 3])))
            placed += 1
        for _ in range(3):
            w = rng.uniform(0.4, 1.0, size=2)
            h = rng.uniform(0.6, 2.0)
            lo = np.array([rng.uniform(lo_x + 0.1, hi_x - w[0] - 0.1), rng.choice([0.1, Y - w[1] - 0.1]), 0.02])
            add(box(lo, lo + [w[0], w[1], h], 3)[0], int(rng.choice([1, 7])))
    first = sum(len(p) for p in parts)
    door, _ = box((X0 + W / 2 - 0.02, y0, 0.0), (X0 + W / 2 + 0.02, y1, zd), 6)
    add(door, 1)
    verts = np.concatenate(parts, axis=0)
    tri_mat = np.concatenate(mats)
    return Scene("door_rooms", verts, tri_mat, absorption_table(n_bands), [src], lis,
                 {"seed": seed, "size": (X1, Y, Z), "door": (first, len(door)), "hinge": (X0 + W / 2, y0)})


def door_verts(scene, angle_deg):
    """the scene's vertices with the door rotated by angle_deg about its hinge (positive: it swings into the listener's
    room); 0 = closed, the door as built"""
    verts = scene.verts.copy()
    if angle_deg == 0:
        return verts
    first, n = scene.meta["door"]
    hx, hy = scene.meta["hinge"]
    a = np.deg2rad(angle_deg)
    d = verts[first:first + n].astype(np.float64)
    dx, dy = d[..., 0] - hx, d[..., 1] - hy
    d[..., 0] = hx + dx * np.cos(a) + dy * np.sin(a)
    d[..., 1] = hy - dx * np.sin(a) + dy * np.cos(a)
    verts[first:first + n] = d.astype(np.float32)
    return verts


def by_name(name, **kw):
    return {"shoebox": shoebox, "furnished_room": furnished_room, "mine_tunnels": mine_tunnels,
            "concert_hall": concert_hall, "door_rooms": door_rooms}[name](**kw)

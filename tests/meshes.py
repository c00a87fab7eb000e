"""Procedural fixture meshes for the meto tokenizer tests.

Same categories as the reference's manual round-trip script (/root/reference/meto/tests/engine.py:39-118:
open patches, closed genus-0, genus-1, inconsistent orientation, strips that exercise L/R runs, fans) plus
multi-component and non-manifold inputs; generated here by code rather than as literal arrays.
All vertices are normalised into the [-0.95, 0.95] cube like ``normalize_mesh(bound=0.95)``.
"""

import numpy as np


def _normalize(v, bound=0.95):
    v = np.asarray(v, dtype=np.float64)
    vmin, vmax = v.min(0), v.max(0)
    return ((v - (vmax + vmin) / 2) * (2 * bound / np.max(vmax - vmin))).astype(np.float32)


def plane():
    v = [[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0]]
    return _normalize(v), np.array([[0, 1, 2], [0, 2, 3]], np.int32)


def tetrahedron():
    v = [[0, 0, 0], [1, 0, 0], [0.5, 1, 0], [0.5, 0.5, 1]]
    return _normalize(v), np.array([[0, 1, 2], [0, 2, 3], [0, 3, 1], [1, 3, 2]], np.int32)


def cube():
    v = [[x, y, z] for z in (0, 1) for y in (0, 1) for x in (0, 1)]
    quads = [(0, 2, 3, 1), (4, 5, 7, 6), (0, 1, 5, 4), (2, 6, 7, 3), (0, 4, 6, 2), (1, 3, 7, 5)]
    f = []
    for a, b, c, d in quads:
        f += [[a, b, c], [a, c, d]]
    return _normalize(v), np.array(f, np.int32)


def strip(n=7, flip=()):
    """Zig-zag triangle strip (long L/R runs); faces listed in ``flip`` get reversed orientation."""
    v = [[i * 0.5, (i % 2), 0.1 * i] for i in range(n + 2)]
    f = []
    for i in range(n):
        tri = [i, i + 1, i + 2] if i % 2 == 0 else [i + 1, i, i + 2]
        if i in flip:
            tri = tri[::-1]
        f.append(tri)
    return _normalize(v), np.array(f, np.int32)


def fan(n=6):
    """Open fan around a centre vertex (the 'split' case when entered from the middle)."""
    v = [[0, 0, 0]] + [[np.cos(a), np.sin(a), 0.2 * np.sin(3 * a)] for a in np.linspace(0, 1.5 * np.pi, n + 1)]
    f = [[0, i + 1, i + 2] for i in range(n)]
    return _normalize(v), np.array(f, np.int32)


def grid(nx=5, ny=4, wavy=True):
    v = [[x, y, (np.sin(x * 1.3) * np.cos(y * 0.7) if wavy else 0)] for y in range(ny + 1) for x in range(nx + 1)]
    f = []
    for y in range(ny):
        for x in range(nx):
            a = y * (nx + 1) + x
            b, c, d = a + 1, a + nx + 2, a + nx + 1
            f += [[a, b, c], [a, c, d]] if (x + y) % 2 == 0 else [[a, b, d], [b, c, d]]
    return _normalize(v), np.array(f, np.int32)


def torus(nu=8, nv=5, R=1.0, r=0.4):
    v, f = [], []
    for i in range(nu):
        for j in range(nv):
            u, w = 2 * np.pi * i / nu, 2 * np.pi * j / nv
            v.append([(R + r * np.cos(w)) * np.cos(u), (R + r * np.cos(w)) * np.sin(u), r * np.sin(w)])
    for i in range(nu):
        for j in range(nv):
            a = i * nv + j
            b = ((i + 1) % nu) * nv + j
            c = ((i + 1) % nu) * nv + (j + 1) % nv
            d = i * nv + (j + 1) % nv
            f += [[a, b, c], [a, c, d]]
    return _normalize(v), np.array(f, np.int32)


def icosphere(sub=1):
    t = (1 + 5 ** 0.5) / 2
    v = [[-1, t, 0], [1, t, 0], [-1, -t, 0], [1, -t, 0], [0, -1, t], [0, 1, t], [0, -1, -t], [0, 1, -t],
         [t, 0, -1], [t, 0, 1], [-t, 0, -1], [-t, 0, 1]]
    f = [[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2], [10, 7, 6],
         [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11], [6, 2, 10],
         [8, 6, 7], [9, 8, 1]]
    v = [list(np.array(p) / np.linalg.norm(p)) for p in v]
    for _ in range(sub):
        cache, nf = {}, []

        def mid(a, b):
            key = (min(a, b), max(a, b))
            if key not in cache:
                m = (np.array(v[a]) + np.array(v[b])) / 2
                v.append(list(m / np.linalg.norm(m)))
                cache[key] = len(v) - 1
            return cache[key]

        for a, b, c in f:
            ab, bc, ca = mid(a, b), mid(b, c), mid(c, a)
            nf += [[a, ab, ca], [b, bc, ab], [c, ca, bc], [ab, bc, ca]]
        f = nf
    return _normalize(v), np.array(f, np.int32)


def annulus(n=10):
    v, f = [], []
    for i in range(n):
        a = 2 * np.pi * i / n
        v += [[0.5 * np.cos(a), 0.5 * np.sin(a), 0], [np.cos(a), np.sin(a), 0.3 * np.cos(2 * a)]]
    for i in range(n):
        a, b = 2 * i, 2 * i + 1
        c, d = 2 * ((i + 1) % n), 2 * ((i + 1) % n) + 1
        f += [[a, b, d], [a, d, c]]
    return _normalize(v), np.array(f, np.int32)


def two_components():
    v1, f1 = tetrahedron()
    v2, f2 = grid(3, 2)
    v = np.concatenate([v1 * 0.4 - 0.5, v2 * 0.4 + 0.5])
    return _normalize(v), np.concatenate([f1, f2 + len(v1)]).astype(np.int32)


def non_manifold():
    """Three triangles sharing one edge."""
    v = [[0, 0, 0], [1, 0, 0], [0.5, 1, 0], [0.5, -1, 0.2], [0.5, 0.3, 1]]
    return _normalize(v), np.array([[0, 1, 2], [1, 0, 3], [0, 1, 4]], np.int32)


def random_soup(seed=3, n=40):
    """Random perturbed grid with some faces deleted and some flipped (holes + orientation repair)."""
    rng = np.random.RandomState(seed)
    v, f = grid(8, 6)
    v = v + rng.uniform(-0.02, 0.02, v.shape).astype(np.float32)
    keep = rng.rand(len(f)) > 0.15
    f = f[keep]
    fl = rng.rand(len(f)) < 0.2
    f[fl] = f[fl][:, ::-1]
    return _normalize(v), f[:n * 2].astype(np.int32)


def all_meshes():
    return {
        'plane': plane(), 'tetrahedron': tetrahedron(), 'cube': cube(), 'strip': strip(), 'strip_flip': strip(flip=(1, 4)),
        'fan': fan(), 'grid': grid(), 'torus': torus(), 'icosphere': icosphere(1), 'icosphere2': icosphere(2),
        'annulus': annulus(), 'two_components': two_components(), 'non_manifold': non_manifold(),
        'random_soup': random_soup(),
    }


def stress_meshes(count=24):
    """Harder tokenizer inputs: holes, flipped faces, shuffled face order, duplicate faces, coincident vertices,
    degenerate triangles, pure random (heavily non-manifold) soups.  Deterministic per index."""
    out = {}
    for seed in range(count):
        r = np.random.RandomState(100 + seed)
        kind = seed % 6
        if kind == 0:
            v, f = random_soup(seed, n=60)
        elif kind == 1:
            v, f = icosphere(3)
            f = f[r.rand(len(f)) > 0.1]
            fl = r.rand(len(f)) < 0.3
            f[fl] = f[fl][:, ::-1]
        elif kind == 2:
            v, f = torus(20, 12)
            f = f[r.permutation(len(f))]
        elif kind == 3:
            v = r.uniform(-0.95, 0.95, (30, 3)).astype(np.float32)
            f = r.randint(0, 30, (80, 3)).astype(np.int32)
        elif kind == 4:
            v, f = grid(6, 6, wavy=False)
            f = np.concatenate([f, f[:10], f[5:9][:, ::-1]])
            v = np.concatenate([v, v[:5]])
        else:
            v, f = grid(30, 30)
            f = f[r.rand(len(f)) > 0.05]
        out[f'stress{seed}'] = (np.ascontiguousarray(v, dtype=np.float32), np.ascontiguousarray(f, dtype=np.int32))
    return out


def random_grids(count=40, seed=2024):
    """Jittered grids with holes, flipped and shuffled faces (every fifth with extra random faces), each with a random bin count:
    yields (index, vertices, faces, bins).  Deterministic for a given seed."""
    rng = np.random.RandomState(seed)
    for it in range(count):
        nx, ny = rng.randint(2, 14, size=2)
        v, f = grid(int(nx), int(ny))
        v = v + rng.uniform(-0.03, 0.03, v.shape).astype(np.float32)
        f = f[rng.rand(len(f)) > rng.uniform(0, 0.3)]
        fl = rng.rand(len(f)) < rng.uniform(0, 0.5)
        f[fl] = f[fl][:, ::-1]
        f = f[rng.permutation(len(f))]
        if it % 5 == 0:                                     # some outright garbage connectivity
            f = np.concatenate([f, rng.randint(0, len(v), (7, 3)).astype(np.int32)])
        v = np.clip(v, -1, 1)
        bins = int(rng.choice([4, 32, 256, 512, 1024]))
        yield it, v, f, bins

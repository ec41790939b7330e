"""Seeded test meshes and rays of the mesh ray cast tests (no GPU needed)."""
import numpy as np


def cube():
    """unit cube [0, 1]^3: 8 vertices, 12 triangles, outward facing"""
    v = np.array([[x, y, z] for x in (0, 1) for y in (0, 1) for z in (0, 1)], np.float32)
    quads = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    t = [[a, b, c] for a, b, c, d in quads] + [[a, c, d] for a, b, c, d in quads]
    return v, np.array(t, np.int32)


def icosphere(subdiv=2):
    """unit icosphere (20 * 4^subdiv triangles, shared vertices)"""
    p = (1 + 5 ** 0.5) / 2
    v = [[-1, p, 0], [1, p, 0], [-1, -p, 0], [1, -p, 0], [0, -1, p], [0, 1, p], [0, -1, -p], [0, 1, -p],
         [p, 0, -1], [p, 0, 1], [-p, 0, -1], [-p, 0, 1]]
    f = [[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2], [10, 7, 6], [7, 1, 8],
         [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11], [6, 2, 10], [8, 6, 7], [9, 8, 1]]
    v = [np.array(x, np.float64) / np.linalg.norm(x) for x in v]
    for _ in range(subdiv):
        mids, nf = {}, []

        def mid(a, b):
            k = (min(a, b), max(a, b))
            if k not in mids:
                m = v[a] + v[b]
                v.append(m / np.linalg.norm(m))
                mids[k] = len(v) - 1
            return mids[k]
        for a, b, c in f:
            ab, bc, ca = mid(a, b), mid(b, c), mid(c, a)
            nf += [[a, ab, ca], [b, bc, ab], [c, ca, bc], [ab, bc, ca]]
        f = nf
    return np.array(v, np.float32), np.array(f, np.int32)


def rays_through(origin, targets):
    """[N, 6] rays from `origin` towards each target (direction = target - origin, not normalised)"""
    t = np.asarray(targets, np.float32)
    o = np.broadcast_to(np.asarray(origin, np.float32), t.shape)
    return np.ascontiguousarray(np.concatenate([o, t - o], 1), dtype=np.float32)


def watertight_rays(v, t, origin, n_random=2000, seed=0):
    """rays from an interior point through every vertex, every edge midpoint and seeded random directions"""
    e = np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]])
    mids = 0.5 * (v[e[:, 0]] + v[e[:, 1]])
    d = np.random.default_rng(seed).normal(size=(n_random, 3)).astype(np.float32)
    return np.concatenate([rays_through(origin, v), rays_through(origin, mids), rays_through(origin, np.asarray(origin, np.float32) + d)])


def soup(n, seed=0, scale=1.0):
    """seeded triangle soup with degenerate, collinear, non-finite and duplicate triangles -> (vertices, triangles)"""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-scale, scale, size=(n, 1, 3))
    v = (c + rng.normal(scale=0.05 * scale, size=(n, 3, 3))).astype(np.float32)
    k = n // 100
    idx = rng.choice(n, size=4 * k, replace=False)
    v[idx[:k], 2] = v[idx[:k], 1]                                     # two equal vertices
    v[idx[k:2 * k], 2] = 2 * v[idx[k:2 * k], 1] - v[idx[k:2 * k], 0]    # (nearly) collinear
    v[idx[2 * k:3 * k], rng.integers(0, 3, k), rng.integers(0, 3, k)] = np.nan
    v[idx[3 * k:], :] = v[rng.choice(n, size=k)]                        # duplicates of other triangles
    return v.reshape(-1, 3), np.arange(3 * n, dtype=np.int32).reshape(n, 3)


def random_rays(n, seed=0, scale=1.5):
    rng = np.random.default_rng(seed)
    o = rng.uniform(-scale, scale, size=(n, 3))
    d = rng.normal(size=(n, 3))
    return np.concatenate([o, d], 1).astype(np.float32)

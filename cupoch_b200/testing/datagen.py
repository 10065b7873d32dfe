"""Synthetic clouds of SURVEY.md section 8d (seeded numpy PCG64, float32).  Shared by tests/ and bench.py."""
import numpy as np


def rot_xyz(rx_deg, ry_deg, rz_deg):
    rx, ry, rz = np.deg2rad([rx_deg, ry_deg, rz_deg])
    Rx = np.array([[1, 0, 0], [0, np.cos(rx), -np.sin(rx)], [0, np.sin(rx), np.cos(rx)]])
    Ry = np.array([[np.cos(ry), 0, np.sin(ry)], [0, 1, 0], [-np.sin(ry), 0, np.cos(ry)]])
    Rz = np.array([[np.cos(rz), -np.sin(rz), 0], [np.sin(rz), np.cos(rz), 0], [0, 0, 1]])
    return Rz @ Ry @ Rx


def gt_transform(angles=(-2.0, 3.0, 5.0), t=(0.02, -0.01, 0.015)):
    """T_gt = Rz(5) Ry(3) Rx(-2), t = (0.02,-0.01,0.015)  (section 8d, config 1)."""
    T = np.eye(4)
    T[:3, :3] = rot_xyz(*angles)
    T[:3, 3] = t
    return T


def uniform_cube(n, seed, lo=(0, 0, 0), hi=(1, 1, 1)):
    rng = np.random.Generator(np.random.PCG64(seed))
    p = rng.random((n, 3), dtype=np.float32)
    return (np.asarray(lo, np.float32) + p * (np.asarray(hi, np.float32) - np.asarray(lo, np.float32))).astype(np.float32)


def unit_normals(n, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    v = rng.standard_normal((n, 3)).astype(np.float32)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    return v.astype(np.float32)


def surface(n, seed, extent=1.0):
    """z = 0.1 sin(4 pi x) cos(4 pi y), x,y ~ U[0,extent); analytic unit normals (config 2)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    xy = rng.random((n, 2)) * extent
    x, y = xy[:, 0], xy[:, 1]
    z = 0.1 * np.sin(4 * np.pi * x) * np.cos(4 * np.pi * y)
    dzdx = 0.4 * np.pi * np.cos(4 * np.pi * x) * np.cos(4 * np.pi * y)
    dzdy = -0.4 * np.pi * np.sin(4 * np.pi * x) * np.sin(4 * np.pi * y)
    nrm = np.stack([-dzdx, -dzdy, np.ones_like(x)], 1)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    return np.stack([x, y, z], 1).astype(np.float32), nrm.astype(np.float32)


def texture(p, seed=None, noise=0.0):
    """smooth colour field in [0,1]^3 (config 5)."""
    x, y = p[:, 0].astype(np.float64), p[:, 1].astype(np.float64)
    c = np.stack([0.5 + 0.4 * np.sin(7 * x) * np.cos(5 * y), 0.5 + 0.4 * np.cos(3 * x + 2 * y),
                  0.5 + 0.4 * np.sin(4 * y - x)], 1)
    if noise > 0:
        rng = np.random.Generator(np.random.PCG64(seed))
        c = c + rng.normal(0, noise, c.shape)
    return np.clip(c, 0, 1).astype(np.float32)


def make_source(target, T_gt, perm_seed, noise_seed, sigma, attrs=()):
    """source = target[perm] moved by T_gt^-1 plus N(0, sigma^2) noise; attrs are permuted and rotated alike."""
    n = len(target)
    perm = np.random.Generator(np.random.PCG64(perm_seed)).permutation(n)
    Ti = np.linalg.inv(T_gt)
    p = target[perm].astype(np.float64) @ Ti[:3, :3].T + Ti[:3, 3]
    if sigma > 0:
        p = p + np.random.Generator(np.random.PCG64(noise_seed)).normal(0, sigma, p.shape)
    out = [p.astype(np.float32)]
    for a, is_vec in attrs:
        b = a[perm]
        if is_vec:
            b = (b.astype(np.float64) @ Ti[:3, :3].T)
        out.append(np.ascontiguousarray(b, np.float32))
    return out if len(out) > 1 else out[0]


def bumps_scene(n, seed, n_bumps=24, extent=1.0):
    """A non-periodic surface for global registration: a height field of seeded Gaussian bumps of varied width and
    height over [0, extent]^2, plus two tilted planes standing on it (float32, [n, 3]).  Unlike surface(), no two
    neighbourhoods repeat, so local descriptors such as FPFH have unambiguous matches."""
    rng = np.random.default_rng(seed)
    c = rng.uniform(0, extent, (n_bumps, 2))
    h = rng.uniform(0.03, 0.12, n_bumps) * extent * rng.choice([-1.0, 1.0], n_bumps)
    w = rng.uniform(0.04, 0.15, n_bumps) * extent
    n_ground = int(n * 0.8)
    xy = rng.uniform(0, extent, (n_ground, 2))
    z = (h[None, :] * np.exp(-((xy[:, None, :] - c[None]) ** 2).sum(-1) / (2 * w[None, :] ** 2))).sum(1)
    ground = np.column_stack([xy, z])
    n_a = (n - n_ground) // 2
    u = rng.uniform(0, 1, (n - n_ground, 2))
    a = u[:n_a]   # tilted plane x = 0.3 extent + 0.4 z, y in [0.1, 0.6] extent
    pa = np.column_stack([0.3 * extent + 0.12 * extent * a[:, 1], (0.1 + 0.5 * a[:, 0]) * extent, 0.3 * extent * a[:, 1]])
    b = u[n_a:]   # tilted plane y = 0.75 extent - 0.32 z, x in [0.45, 0.95] extent
    pb = np.column_stack([(0.45 + 0.5 * b[:, 0]) * extent, 0.75 * extent - 0.08 * extent * b[:, 1], 0.25 * extent * b[:, 1]])
    return np.concatenate([ground, pa, pb]).astype(np.float32)

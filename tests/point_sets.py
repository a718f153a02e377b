"""Point sets for the per-point projection tests: the host build of the point function
(test_host_abi.py) and the device kernels (test_gpu_projection_points.py) take the same points.
Each set aims at one place where the pixel assignment can go wrong: bin edges, the |x| = |y| octant
lines, coordinates next to or on the vertical axis, signed zeros, the range limits and non-finite
or overflowing coordinates. All generators return contiguous float32 (N, 3) arrays."""
import numpy as np

from oracle import nsc_oracle as orc

F32 = np.float32


def _kept_ranges(rng, n, cfg):
    """Ranges strictly inside [min_range, max_range] (min_range 0 -> from 0.3)."""
    lo, hi = max(cfg.min_range, 0.3), cfg.max_range
    return rng.uniform(lo + 1e-3 * (hi - lo), hi - 1e-3 * (hi - lo), n)


def from_angles(az, el, r):
    """float64 (azimuth as atan2(y, x), elevation, range) -> float32 xyz."""
    return np.stack([r * np.cos(el) * np.cos(az), r * np.cos(el) * np.sin(az), r * np.sin(el)], 1).astype(F32)


def uniform_sphere(rng, n, lo=0.3, hi=120.0):
    """Directions uniform over the sphere, ranges log-uniform in [lo, hi]."""
    v = rng.normal(size=(n, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    return np.ascontiguousarray((v * np.exp(rng.uniform(np.log(lo), np.log(hi), n))[:, None]).astype(F32))


def edge_points(rng, cfg, n, offset=1.01e-5):
    """About n points `offset` rad on either side of every column edge and every inner row edge:
    outside the 1e-5 rad excuse, so they must land in the oracle's pixel."""
    el_lo, el_hi = float(cfg.el_min), float(cfg.el_max)
    cw = 2 * np.pi / cfg.n_azimuth
    rw = (el_hi - el_lo) / cfg.n_elevation
    n_col = n if cfg.n_elevation == 1 else n // 2
    k = rng.integers(0, cfg.n_azimuth, n_col)
    az = k * cw - np.pi + rng.choice([-offset, offset], n_col)       # the oracle's azimuth is atan2 + pi
    el = rng.uniform(max(el_lo, -1.5), min(el_hi, 1.5), n_col)
    parts = [from_angles(az, el, _kept_ranges(rng, n_col, cfg))]
    if cfg.n_elevation > 1:
        m = n - n_col
        q = rng.integers(1, cfg.n_elevation, m)
        el = el_lo + q * rw + rng.choice([-offset, offset], m)
        parts.append(from_angles(rng.uniform(-np.pi, np.pi, m), el, _kept_ranges(rng, m, cfg)))
    return np.ascontiguousarray(np.concatenate(parts))


def octant_lines(rng, n, cfg):
    """|x| == |y| exactly in float32: the azimuth is an odd multiple of 45 degrees."""
    r, el = _kept_ranges(rng, n, cfg), rng.uniform(-1.5, 1.5, n)
    a = (r * np.cos(el) / np.sqrt(2)).astype(F32)
    s = rng.choice([-1, 1], (n, 2)).astype(F32)
    return np.ascontiguousarray(np.stack([s[:, 0] * a, s[:, 1] * a, (r * np.sin(el)).astype(F32)], 1))


def near_axis(rng, n, cfg):
    """|x| and |y| in [1e-45, 1e-20] (subnormals included), all four sign quadrants, z inside the
    range limits: points next to the vertical axis, whose column is atan2(y, x) all the same. Half
    of them with independent |x|, |y|; half with |y| / |x| in [0.1, 10], an azimuth away from the
    axes."""
    h = n // 2
    ax = 10.0 ** rng.uniform(-45, -20, n)
    ay = np.concatenate([10.0 ** rng.uniform(-45, -20, h), ax[h:] * 10.0 ** rng.uniform(-1, 1, n - h)])
    s = rng.choice([-1, 1], (n, 3))
    z = s[:, 2] * _kept_ranges(rng, n, cfg)
    return np.ascontiguousarray(np.stack([s[:, 0] * ax, s[:, 1] * ay, z], 1).astype(F32))


def signed_zeros(cfg):
    """Points on the x, y and z axes and above them: +0, -0, +a, -a in x and y (one
    of them a zero) with +0, -0, +-b in z (a, b ranges inside the limits), so the azimuth wrap
    (x < 0, y = +-0) is there too. The origin is left out: it has no direction, and it is kept only
    when min_range is 0. (|x| = |y| points lie on column edges: octant_lines.)"""
    a = F32(0.5 * (max(cfg.min_range, 0.3) + cfg.max_range))
    b = F32(max(cfg.min_range, 0.3) * 1.5)
    xy = [F32(0.0), F32(-0.0), a, -a]
    zs = [F32(0.0), F32(-0.0), b, -b]
    pts = [(x, y, z) for x in xy for y in xy for z in zs if (x == 0 or y == 0) and (x != 0 or y != 0 or z != 0)]
    return np.array(pts, F32)


ADVERSARIAL = np.array([np.nan, -np.nan, np.inf, -np.inf, 0.0, -0.0, 1e-45, -1e-45, 1e-40, -3e-39, 1e-30,
                        1e38, -1e38, 3.4e38, 2e19, -1.9e19, 1.8e19, 5e18, 2.0, -7.5], F32)


def adversarial(rng, n_base, cfg):
    """NaN / +-Inf, subnormals, +-1e38 and coordinates whose squares overflow, in each coordinate
    of in-range base points alone and in every triple of such values."""
    base = from_angles(rng.uniform(-np.pi, np.pi, n_base), rng.uniform(-1.0, 1.0, n_base),
                       _kept_ranges(rng, n_base, cfg))
    parts = []
    for c in range(3):
        p = np.repeat(base, len(ADVERSARIAL), 0)
        p[:, c] = np.tile(ADVERSARIAL, n_base)
        parts.append(p)
    g = np.stack(np.meshgrid(ADVERSARIAL, ADVERSARIAL, ADVERSARIAL, indexing="ij"), -1).reshape(-1, 3)
    parts.append(g)
    return np.ascontiguousarray(np.concatenate(parts))


def range_limits(rng, cfg, n_ulps=6):
    """Points a few float32 ulps on either side of min_range and max_range, and far outside them."""
    rs = []
    for r0 in (cfg.min_range, cfg.max_range):
        v = F32(r0)
        for _ in range(n_ulps):
            v = np.nextafter(v, F32(0))
        for _ in range(2 * n_ulps + 1):
            rs.append(v)
            v = np.nextafter(v, F32(np.inf))
    rs = np.array(rs * 40, np.float64)
    far = np.concatenate([rng.uniform(0.0, max(cfg.min_range, 1e-3), 500), rng.uniform(cfg.max_range * 1.01, 1e4, 500)])
    r = np.concatenate([rs, far])
    return from_angles(rng.uniform(-np.pi, np.pi, len(r)), rng.uniform(-1.5, 1.5, len(r)), r)


def oracle_pixels(pts, cfg):
    """Per point: kept (bool), the oracle's row / column / float32 range (-1 / -1 / nan if
    dropped) and the distances to the nearest column / row edge (float64 rad)."""
    n = len(pts)
    with np.errstate(over="ignore", invalid="ignore"):      # overflowing squares are part of the sets
        s = orc.spherical(pts, cfg)
    kept = np.zeros(n, bool)
    kept[s["kept"]] = True
    row, col = np.full(n, -1, np.int64), np.full(n, -1, np.int64)
    rng = np.full(n, np.nan, F32)
    row[s["kept"]], col[s["kept"]], rng[s["kept"]] = s["row"], s["col"], s["range"]
    d_az, d_el = orc.edge_distance(pts, cfg)
    return kept, row, col, rng, d_az, d_el


def across_edges(pts, cfg, row, col):
    """The row and the column across each point's nearest row / column edge (rows clamp: the outer
    FOV limits are not edges; columns wrap mod n_azimuth)."""
    p = np.asarray(pts, np.float64)
    with np.errstate(invalid="ignore"):
        az = np.arctan2(p[:, 1], p[:, 0]) + np.pi
        el = np.arctan2(p[:, 2], np.sqrt(p[:, 0] ** 2 + p[:, 1] ** 2))
    W, E = cfg.n_azimuth, cfg.n_elevation
    m = np.nan_to_num(np.round(az / (2 * np.pi / W))).astype(np.int64)
    col_x = np.where(col == m % W, (m - 1) % W, m % W)
    rw = (float(cfg.el_max) - float(cfg.el_min)) / E
    q = np.clip(np.nan_to_num(np.round((el - float(cfg.el_min)) / rw)), 1, max(E - 1, 1)).astype(np.int64)
    row_x = np.clip(np.where(row == q, q - 1, q), 0, E - 1)
    return row_x, col_x
